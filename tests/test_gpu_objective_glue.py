"""GPU tests of the glue kernels of the fused objective (csrc/objective_fused.cu) and of the objective paths that the
whole-objective comparisons do not reach.

  * dmh_disp_grad in each of its launch regimes (restated on the host), every element against a float64 reference
    within a rounding bound derived from the number of accumulated taps;
  * dmh_smooth_fused (C = 3 and C = 1) and dmh_objective_finish against float64, element by element;
  * the public objective with six scales and with per-scale upstream gradients (`loss/s` weighted separately);
  * the IEEE-division builds of the photometric kernels, which run when a size is first seen inside a CUDA-graph
    capture.

Rounding bounds: with u = 2^-24, a value computed as a sum of terms that each pass through at most k roundings is
within k * u * sum|terms| of the exact sum (first order).  A dropped or duplicated term moves a value by |term|,
far beyond that bound, which a max-relative check over the whole tensor would not see.
"""
import ctypes as C
import re

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from depthmodelhardening_b200 import synth
from oracle import photometric as OP
from tests.util import assert_close, assert_grad_close

pytestmark = pytest.mark.gpu
U = 2.0 ** -24
TOL = 1e-5
DEV = "cuda:0"


@pytest.fixture(scope="module")
def lib():
    from depthmodelhardening_b200 import _lib
    return _lib.load()


def _call(rc, what):
    from depthmodelhardening_b200._lib import check
    check(rc, what)


def _ptr(t):
    from depthmodelhardening_b200._lib import ptr
    return ptr(t)


def _stream():
    from depthmodelhardening_b200._lib import stream
    return stream()


def _at_offset(src, off):
    """A contiguous copy of `src` on the device that starts `off` floats into its allocation (off = 1: 4-byte but not
    16-byte aligned)."""
    base = torch.empty(src.numel() + off, device=DEV)
    v = base[off:off + src.numel()].view(src.shape)
    v.copy_(src)
    return v


def _assert_within(got, ref, bound, what, mask=None):
    """|got - ref| <= bound for every element (float64 arithmetic); `mask` selects the elements compared."""
    got = got.double()
    assert torch.isfinite(got).all(), "%s: non-finite elements" % what
    err = (got - ref).abs()
    bad = err > bound
    if mask is not None:
        bad &= mask
    n = int(bad.sum())
    if n:
        idx = tuple(int(i) for i in bad.nonzero()[0])
        ratio = float((err / bound.clamp_min(1e-300))[bad].max())
        raise AssertionError("%s: %d of %d elements beyond the rounding bound (worst %.3g x the bound; first at %s: "
                             "got %r, expected %r, bound %.3g)" % (what, n, bad.numel(), ratio, idx, float(got[idx]),
                                                                   float(ref[idx]), float(bound[idx])))


# ----------------------------------------------------------------------------- dmh_disp_grad
def _up_weights(n_out, n_in):
    """(n_out, n_in) float64 matrix of F.interpolate(bilinear, align_corners=False) weights with the kernels' fp32
    arithmetic (dmh_common.cuh up_tap, compiled to src = fma(in/out, dst + 0.5, -0.5): one rounding), l1 = src - i0,
    l0 = 1 - l1, and a tap clamped at the last pixel counts l0 + l1 (added in fp32)."""
    sc = np.float32(n_in) / np.float32(n_out)
    t = np.arange(n_out, dtype=np.float32) + np.float32(0.5)
    src = (np.float64(sc) * t.astype(np.float64) - 0.5).astype(np.float32)     # exact product, one rounding
    src = np.maximum(src, np.float32(0.0))
    i0 = np.minimum(src.astype(np.int64), n_in - 1)
    i1 = np.where(i0 < n_in - 1, i0 + 1, i0)
    l1 = (src - i0.astype(np.float32)).astype(np.float32)
    l0 = (np.float32(1.0) - l1).astype(np.float32)
    A = np.zeros((n_out, n_in))
    r = np.arange(n_out)
    same = i0 == i1
    A[r, i0] = np.where(same, (l0 + l1).astype(np.float32), l0)
    A[r[~same], i1[~same]] = l1[~same]
    return A


def _dg_regime(h, w, H, W, p_g, p_gn, p_out):
    """Host restatement of dmh_disp_grad's kernel choice (objective_fused.cu)."""
    R = H // h if (H % h == 0 and W % w == 0 and H // h == W // w) else 0
    if R > 1 and (p_g % 16 != 0 or W % 4 != 0):
        R = 0
    if R == 1 and (h * w) % 4 == 0 and p_g % 16 == 0 and p_out % 16 == 0 and (p_gn is None or p_gn % 16 == 0):
        return "same_float4"
    if R == 1:
        return "same_scalar"
    if R in (2, 4, 8):
        return "tall%d" % R
    return "generic"


# (B, h, w, H, W, float offsets of (G, gN, output), regime the host restatement must pick)
DG_CASES = [
    (2, 40, 64, 40, 64, (0, 0, 0), "same_float4"),
    (32, 320, 1024, 320, 1024, (0, 0, 0), "same_float4"),      # the benchmark's scale 0
    (2, 16, 1, 16, 1, (0, 0, 0), "same_float4"),               # w = 1
    (3, 33, 37, 33, 37, (0, 0, 0), "same_scalar"),             # h*w % 4 != 0
    (2, 40, 64, 40, 64, (1, 0, 0), "same_scalar"),             # G 4-byte aligned
    (2, 40, 64, 40, 64, (0, 1, 0), "same_scalar"),             # gN 4-byte aligned
    (2, 40, 64, 40, 64, (0, 0, 1), "same_scalar"),             # output 4-byte aligned
    (1, 1, 1, 1, 1, (0, 0, 0), "same_scalar"),                 # h = w = 1
    (2, 80, 100, 160, 200, (0, 0, 0), "tall2"),                # several tiles in x and y
    (2, 25, 36, 50, 72, (0, 0, 0), "tall2"),                   # h % 32, w % 32 != 0
    (2, 18, 50, 72, 200, (0, 0, 0), "tall4"),                  # h % 16, w % 32 != 0
    (2, 1, 10, 4, 40, (0, 0, 0), "tall4"),                     # h = 1
    (2, 9, 25, 72, 200, (0, 0, 0), "tall8"),                   # h % 8, w % 32 != 0
    (32, 40, 128, 320, 1024, (0, 0, 0), "tall8"),              # the benchmark's scale 3
    (2, 25, 36, 50, 72, (1, 0, 0), "generic"),                 # R = 2 with a 4-byte aligned G
    (2, 11, 13, 33, 39, (0, 0, 0), "generic"),                 # R = 3
    (1, 5, 7, 80, 112, (0, 0, 0), "generic"),                  # R = 16
    (1, 3, 5, 96, 160, (0, 0, 0), "generic"),                  # R = 32
    (2, 17, 19, 96, 160, (0, 0, 0), "generic"),                # non-integer factors
    (2, 24, 20, 96, 160, (0, 0, 0), "generic"),                # H/h = 4, W/w = 8
    (2, 12, 21, 24, 42, (0, 0, 0), "generic"),                 # R = 2, W % 4 != 0
    (2, 1, 40, 8, 80, (0, 0, 0), "generic"),                   # h = 1
    (2, 12, 1, 24, 2, (0, 0, 0), "generic"),                   # w = 1
]

# upstream scalars: (g_total, g_scale, g_smooth, with gN)
DG_FORMS = {"g_total": (True, False, False, True), "g_scale": (False, True, False, True),
            "g_total+g_scale": (True, True, False, True), "g_smooth": (True, False, True, True),
            "no gN": (True, True, False, False)}


def test_disp_grad_case_table_reaches_every_regime():
    regimes = {_dg_regime(h, w, H, W, 4 * og, 4 * on, 4 * oo) for _, h, w, H, W, (og, on, oo), _ in DG_CASES}
    assert regimes == {"same_float4", "same_scalar", "tall2", "tall4", "tall8", "generic"}
    for _, h, w, H, W, (og, on, oo), want in DG_CASES:
        assert _dg_regime(h, w, H, W, 4 * og, 4 * on, 4 * oo) == want, (h, w, H, W)


@pytest.mark.parametrize("B,h,w,H,W,offs,regime", DG_CASES)
def test_disp_grad_every_element_vs_fp64(lib, B, h, w, H, W, offs, regime):
    """d(objective)/d(disp_s) = up * (interpolate^T(G) + sw * (gN * inv_m - corr)), or g_smooth * sw * (...) +
    up * interpolate^T(G) in the depth-hints form, with up = g_total / S + g_scale.  Bound per element:
    k * u * (|up| * interpolate^T(|G|) + |sw| * (|gN * inv_m| + |corr|) * (|up| or |g_smooth|)), k = ntx + nty + 8:
    a tap passes through at most ntx roundings in its row sum (plus the tall tile's add of the two chunk halves) and
    nty in the column sum, then acc + sm, the multiplication by up, the two roundings of up and the two of sm.  The
    reference uses the kernels' fp32 interpolation weights (the weights ATen's fp32 up-sampling uses), checked against
    float64 F.interpolate."""
    og, on, oo = offs
    gen = torch.Generator().manual_seed(1000 + h * 7 + w * 13 + H + W + og + 2 * on + 3 * oo)
    G = torch.randn(B, 1, H, W, generator=gen)
    gN = torch.randn(B, 1, h, w, generator=gen)
    scal = torch.stack([0.5 + 3 * torch.rand(B, generator=gen), torch.randn(B, generator=gen)], 1).contiguous()
    sw = float(np.float32(0.37))
    S = 3
    inv_S = float(np.float32(1.0 / S))
    vals = {"g_total": 1.7, "g_scale": -0.6, "g_smooth": 2.3}
    Gd, gNd = _at_offset(G.to(DEV), og), _at_offset(gN.to(DEV), on)
    scald = scal.to(DEV)
    new_out = lambda: _at_offset(torch.full((B, 1, h, w), float("nan"), device=DEV), oo)
    assert _dg_regime(h, w, H, W, Gd.data_ptr(), gNd.data_ptr(), new_out().data_ptr()) == regime
    Ay = torch.from_numpy(_up_weights(H, h)).to(DEV)
    Ax = torch.from_numpy(_up_weights(W, w)).to(DEV)
    G64 = G.double().to(DEV)[:, 0]
    acc = torch.einsum("Yy,bYX,Xx->byx", Ay, G64, Ax)
    acc_abs = torch.einsum("Yy,bYX,Xx->byx", Ay, G64.abs(), Ax)
    # the restated weights are ATen's: float64 F.interpolate's transpose agrees to the fp32 rounding of lambda
    x = torch.zeros(B, 1, h, w, dtype=torch.float64, device=DEV, requires_grad=True)
    F.interpolate(x, [H, W], mode="bilinear", align_corners=False).backward(G64[:, None])
    assert float((x.grad[:, 0] - acc).abs().max()) <= 1e-5 * float(acc_abs.max())
    ntx = int((Ax != 0).sum(0).max())
    nty = int((Ay != 0).sum(0).max())
    k = ntx + nty + 8
    inv_m = scal[:, 0].double().to(DEV).view(B, 1, 1)
    corr = scal[:, 1].double().to(DEV).view(B, 1, 1)
    gN64 = gN.double().to(DEV)[:, 0]
    for form, (has_t, has_s, has_sm, has_n) in DG_FORMS.items():
        gt = torch.tensor([vals["g_total"]], device=DEV) if has_t else None
        gs = torch.tensor([vals["g_scale"]], device=DEV) if has_s else None
        gsm = torch.tensor([vals["g_smooth"]], device=DEV) if has_sm else None
        out = new_out()
        _call(lib.dmh_disp_grad(_ptr(Gd), _ptr(gNd) if has_n else None, _ptr(scald), sw, _ptr(gt), _ptr(gs), _ptr(gsm),
                                inv_S, B, h, w, H, W, _ptr(out), _stream()), "disp_grad")
        torch.cuda.synchronize()
        ut = float(np.float32(vals["g_total"])) * inv_S if has_t else 0.0
        us = float(np.float32(vals["g_scale"])) if has_s else 0.0
        up, up_abs = ut + us, abs(ut) + abs(us)
        if has_n:
            sm = sw * (gN64 * inv_m - corr)
            sm_abs = sw * ((gN64 * inv_m).abs() + corr.abs())
        else:
            sm = sm_abs = torch.zeros_like(acc)
        if has_sm:
            g_sm = float(np.float32(vals["g_smooth"]))
            ref = g_sm * sm + up * acc
            terms = abs(g_sm) * sm_abs + up_abs * acc_abs
        else:
            ref = up * (acc + sm)
            terms = up_abs * (acc_abs + sm_abs)
        _assert_within(out[:, 0], ref, k * U * terms, "%s %s (%d,%d)->(%d,%d)" % (regime, form, h, w, H, W))


def test_disp_grad_refuses_missing_upstream(lib):
    G = torch.zeros(1, 1, 8, 8, device=DEV)
    out = torch.empty(1, 1, 4, 4, device=DEV)
    assert lib.dmh_disp_grad(_ptr(G), None, None, 1.0, None, None, None, 1.0, 1, 4, 4, 8, 8, _ptr(out), _stream()) != 0


# ----------------------------------------------------------------------------- dmh_smooth_fused + dmh_objective_finish
def _smooth_inputs(B, C_, h, w, seed):
    gen = torch.Generator().manual_seed(seed)
    d = 0.05 + 0.4 * torch.rand(B, 1, h, w, generator=gen)
    if h >= 4 and w >= 6:
        d[:, :, 1:4, 2:6] = 0.25                         # exactly equal neighbours: sgn(0) = 0 on both sides
    img = torch.rand(B, C_, h, w, generator=gen)
    return d.contiguous(), img.contiguous()


def _smooth_ref(d, img):
    """float64 restatement of oracle/photometric.py normalised_smooth_loss and its gradient w.r.t. the normalised
    disparity, plus the quantities the rounding bounds need."""
    B, C_, h, w = img.shape
    d64, i64 = d.double(), img.double()
    m = d64.mean((2, 3), keepdim=True) + 1e-7
    dn = d64 / m
    ex = torch.exp(-(i64[..., :, :-1] - i64[..., :, 1:]).abs().mean(1, keepdim=True))
    ey = torch.exp(-(i64[..., :-1, :] - i64[..., 1:, :]).abs().mean(1, keepdim=True))
    dx, dy = dn[..., :, :-1] - dn[..., :, 1:], dn[..., :-1, :] - dn[..., 1:, :]
    inx, iny = 1.0 / (B * h * (w - 1)), 1.0 / (B * (h - 1) * w)
    loss = (dx.abs() * ex).sum() * inx + (dy.abs() * ey).sum() * iny
    gx, gy = torch.sign(dx) * ex * inx, torch.sign(dy) * ey * iny
    g = torch.zeros_like(dn)
    g[..., :, :-1] += gx; g[..., :, 1:] -= gx; g[..., :-1, :] += gy; g[..., 1:, :] -= gy
    T = torch.zeros_like(dn)                             # sum of |terms| of each gradient element
    T[..., :, :-1] += ex * inx; T[..., :, 1:] += ex * inx; T[..., :-1, :] += ey * iny; T[..., 1:, :] += ey * iny
    # edges whose fp32 sign may differ: neighbours that are not equal but within a few ulp after normalisation
    # (fl(d_j * inv_m) is monotone in d_j, so the fp32 sign is either the fp64 sign or 0)
    tx = (d64[..., :, :-1] != d64[..., :, 1:]) & (dx.abs() <= 4 * U * torch.maximum(dn[..., :, :-1], dn[..., :, 1:]))
    ty = (d64[..., :-1, :] != d64[..., 1:, :]) & (dy.abs() <= 4 * U * torch.maximum(dn[..., :-1, :], dn[..., 1:, :]))
    tie = torch.zeros_like(dn, dtype=torch.bool)
    tie[..., :, :-1] |= tx; tie[..., :, 1:] |= tx; tie[..., :-1, :] |= ty; tie[..., 1:, :] |= ty
    tie_corr = 2 * ((ex * inx * (d64[..., :, :-1] - d64[..., :, 1:]).abs() * tx).sum((1, 2, 3)) +
                    (ey * iny * (d64[..., :-1, :] - d64[..., 1:, :]).abs() * ty).sum((1, 2, 3)))
    loss_terms = ((dx.abs() + 2 * (dn[..., :, :-1] + dn[..., :, 1:])) * ex).sum() * inx + \
                 ((dy.abs() + 2 * (dn[..., :-1, :] + dn[..., 1:, :])) * ey).sum() * iny
    corr = (g * d64).sum((1, 2, 3)) / (h * w) / m.view(B) ** 2
    return dict(loss=float(loss), loss_terms=float(loss_terms), g=g, T=T, tie=tie, inv_m=1.0 / m.view(B), corr=corr,
                corr_terms=((g * d64).abs().sum((1, 2, 3)), (d64.abs() * T).sum((1, 2, 3)), tie_corr))


def _run_smooth_and_finish(lib, B, C_, sizes, seed):
    """dmh_smooth_fused per scale, then dmh_objective_finish with zero photometric partials: each per-scale loss is
    the weighted smoothness term alone."""
    S = len(sizes)
    ins, wss, gNs = [], [], []
    for s, (h, w) in enumerate(sizes):
        d, img = _smooth_inputs(B, C_, h, w, seed + s)
        dd, imd = d.to(DEV), img.to(DEV)
        ws = torch.full((lib.dmh_smooth_fused_workspace_floats(B, h, w),), float("nan"), device=DEV)
        gN = torch.full((B, 1, h, w), float("nan"), device=DEV)
        _call(lib.dmh_smooth_fused(_ptr(dd), _ptr(imd), B, C_, h, w, _ptr(ws), _ptr(gN), _stream()), "smooth_fused")
        ins.append((d, img)); wss.append(ws); gNs.append(gN)
    sw = [float(np.float32(1e-3 / 2 ** s)) for s in range(S)]
    zeros = [torch.zeros(5, device=DEV) for _ in range(S)]
    scal = torch.full((S, B, 2), float("nan"), device=DEV)
    losses = torch.full((S + 1,), float("nan"), device=DEV)
    fin = torch.empty(lib.dmh_objective_finish_workspace_bytes(S, B), device=DEV, dtype=torch.uint8)
    from depthmodelhardening_b200._lib import ptr_array
    _call(lib.dmh_objective_finish(S, B, ptr_array(wss), (C.c_int * S)(*[h for h, _ in sizes]),
                                   (C.c_int * S)(*[w for _, w in sizes]), ptr_array(zeros), (C.c_int * S)(*([5] * S)),
                                   (C.c_float * S)(*sw), 1.0, _ptr(fin), _ptr(scal), _ptr(losses), _stream()), "finish")
    torch.cuda.synchronize()
    return ins, gNs, scal.cpu(), losses.cpu(), sw


SMOOTH_CASES = [(2, 3, [(2, 2)]), (2, 3, [(32, 128), (33, 129), (32, 129), (33, 128)]),
                (2, 3, [(40, 70)]),                        # w % 4 != 0: scalar loads
                (3, 3, [(33, 37), (31, 70)]),              # h*w % 4 != 0: images b > 0 misaligned for the float4 mean
                (32, 3, [(320, 1024), (160, 512), (80, 256), (40, 128)]),   # the benchmark's scales at B = 32
                (2, 1, [(33, 129), (40, 72), (2, 2)])]     # C = 1


@pytest.mark.parametrize("B,C_,sizes", SMOOTH_CASES)
def test_smooth_fused_and_finish_vs_fp64(lib, B, C_, sizes):
    """Smoothness loss, gradient w.r.t. the normalised disparity, 1/(mean+1e-7) and the normalisation-backward
    correction against float64.  Bounds (u = 2^-24):
      gN        k_g = C + 12: the edge weight exp2(-sum_c|dI| log2e / C) (C - 1 adds, C subtractions, two products,
                ex2.approx: <= 2^-22) and the gradient's subtraction, product, FMA and the fp32 1/(B h (w-1));
                edges whose two normalised disparities are within 4 ulp but not equal may flip sgn() and are excluded;
      inv_m     k_m = ceil(hw / 16384) + 24: a thread's sequential sum, the float4 pair sums, the block and warp
                trees, the division by hw, + 1e-7 and the reciprocal (all terms positive);
      loss      k_l = 16 + 8 + (C + 6) + k_m + 6 against sum(e * (|dx| + 2 (|dn_j| + |dn_j+1|))): 16 terms per lane,
                the reductions, the edge weight, the fp32 normalisation and the final conversion;
      corr      inv_m^2 / hw * (k_g u sum|d| T + 24 u sum|g d| + the flipped-edge term) + (2 k_m + 3) u |corr|."""
    ins, gNs, scal, losses, sw = _run_smooth_and_finish(lib, B, C_, sizes, seed=700 + B + C_)
    S = len(sizes)
    total_ref = 0.0
    for s, (h, w) in enumerate(sizes):
        d, img = ins[s]
        r = _smooth_ref(d, img)
        k_g, k_m = C_ + 12, -(-h * w // 16384) + 24
        k_l = 16 + 8 + (C_ + 6) + k_m + 6
        tie = r["tie"]
        assert float(tie.double().mean()) < 1e-2, "too many near-tied edges for a meaningful comparison"
        _assert_within(gNs[s].cpu(), r["g"], k_g * U * r["T"], "gN scale %d (%dx%d, C=%d)" % (s, h, w, C_), mask=~tie)
        _assert_within(scal[s, :, 0], r["inv_m"], k_m * U * r["inv_m"], "1/(mean+eps) scale %d" % s)
        gd, dT, tie_c = r["corr_terms"]
        inv_m2 = r["inv_m"] ** 2
        cb = inv_m2 / (h * w) * (k_g * U * dT + 24 * U * gd + tie_c) + (2 * k_m + 3) * U * r["corr"].abs()
        _assert_within(scal[s, :, 1], r["corr"], cb, "corr scale %d" % s)
        lref = sw[s] * r["loss"]
        lb = sw[s] * k_l * U * r["loss_terms"]
        assert abs(float(losses[s]) - lref) <= lb, "loss/%d: %r vs %r (bound %.3g)" % (s, float(losses[s]), lref, lb)
        total_ref += lref
    assert abs(float(losses[S]) - total_ref / S) <= 1e-6 * abs(total_ref / S)


def _finish_inputs(S, B, seed):
    gen = torch.Generator().manual_seed(seed)
    pool = [(2, 2), (33, 129), (40, 128), (7, 300), (64, 64), (320, 1024), (3, 5), (160, 512)]
    sizes = [pool[(s * 3 + B) % len(pool)] for s in range(S)]
    ns = [7 * B + 3, max(B - 1, 1), 12345, 1, 3 * B, 0 if B > 1 else 2, 65, 4097]
    ws, parts, pns = [], [], []
    for s, (h, w) in enumerate(sizes):
        nb = -(-w // 128) * -(-h // 32)
        mean_p = torch.rand(B, 64, generator=gen) * 3.0
        sm_p = torch.rand(B, nb, 3, generator=gen)
        sm_p[..., 2] = torch.randn(B, nb, generator=gen)
        ws.append(torch.cat([mean_p.reshape(-1), sm_p.reshape(-1)]))
        n = ns[s]
        parts.append(torch.rand(max(n, 1), generator=gen) * 10.0)
        pns.append(n)
    sw = [float(np.float32(x)) for x in torch.rand(S, generator=gen) * 1e-3]
    return sizes, ws, parts, pns, sw


@pytest.mark.parametrize("S", [1, 4, 5, 8])
@pytest.mark.parametrize("B", [1, 31, 32, 33, 65])
def test_objective_finish_vs_fp64(lib, S, B):
    """dmh_objective_finish on random partial sums: the per-scale losses and their mean equal a float64 sum of the
    same partials to fp32 rounding (u |x| + a float64 allowance), the image scalars within their fp32 chains; photo
    partial counts not divisible by B and smaller than B; the last-CTA ticket is reset (a second call on the same
    workspace gives the same bits)."""
    from depthmodelhardening_b200._lib import ptr_array
    sizes, ws, parts, pns, sw = _finish_inputs(S, B, seed=900 + 10 * S + B)
    den = 12345.0
    wsd = [t.to(DEV) for t in ws]
    pd = [t.to(DEV) for t in parts]
    fin = torch.empty(lib.dmh_objective_finish_workspace_bytes(S, B), device=DEV, dtype=torch.uint8)
    outs = []
    for _ in range(2):
        scal = torch.full((S, B, 2), float("nan"), device=DEV)
        losses = torch.full((S + 1,), float("nan"), device=DEV)
        _call(lib.dmh_objective_finish(S, B, ptr_array(wsd), (C.c_int * S)(*[h for h, _ in sizes]),
                                       (C.c_int * S)(*[w for _, w in sizes]), ptr_array(pd), (C.c_int * S)(*pns),
                                       (C.c_float * S)(*sw), den, _ptr(fin), _ptr(scal), _ptr(losses), _stream()),
              "finish")
        torch.cuda.synchronize()
        outs.append((scal.cpu(), losses.cpu()))
    assert torch.equal(outs[0][0].view(torch.int32), outs[1][0].view(torch.int32))
    assert torch.equal(outs[0][1].view(torch.int32), outs[1][1].view(torch.int32))
    scal, losses = outs[0]
    tot, tot_terms = 0.0, 0.0
    for s, (h, w) in enumerate(sizes):
        hw = h * w
        mp = ws[s][:B * 64].double().view(B, 64)
        sp = ws[s][B * 64:].double().view(B, -1, 3)
        inv_m = 1.0 / (mp.sum(1) / hw + 1e-7)
        corr = sp[..., 2].sum(1) / hw * inv_m ** 2
        _assert_within(scal[s, :, 0], inv_m, 10 * U * inv_m, "inv_m scale %d" % s)
        cterms = sp[..., 2].abs().sum(1) / hw * inv_m ** 2
        _assert_within(scal[s, :, 1], corr, 23 * U * corr.abs() + 2.0 ** -45 * cterms, "corr scale %d" % s)
        ph = parts[s][:pns[s]].double().sum()
        inx, iny = 1.0 / (B * h * (w - 1)), 1.0 / (B * (h - 1) * w)
        loss = float(ph / den + sw[s] * (sp[..., 0].sum() * inx + sp[..., 1].sum() * iny))
        assert abs(float(losses[s]) - loss) <= U * abs(loss) + 2.0 ** -45 * loss, \
            "loss/%d (S=%d, B=%d, photo_n=%d): %r vs float64 %r" % (s, S, B, pns[s], float(losses[s]), loss)
        tot += loss
    assert abs(float(losses[S]) - tot / S) <= U * abs(tot / S) + 2.0 ** -45 * tot


def test_objective_finish_refuses_nine_scales(lib):
    from depthmodelhardening_b200._lib import ptr_array
    S, B = 9, 2
    ws = [torch.zeros(B * 64 + 3 * B, device=DEV) for _ in range(S)]
    fin = torch.empty(lib.dmh_objective_finish_workspace_bytes(S, B), device=DEV, dtype=torch.uint8)
    scal = torch.empty(S, B, 2, device=DEV)
    losses = torch.empty(S + 1, device=DEV)
    rc = lib.dmh_objective_finish(S, B, ptr_array(ws), (C.c_int * S)(*([2] * S)), (C.c_int * S)(*([2] * S)),
                                  ptr_array(ws), (C.c_int * S)(*([1] * S)), (C.c_float * S)(*([1.0] * S)), 1.0,
                                  _ptr(fin), _ptr(scal), _ptr(losses), _stream())
    assert rc != 0


# ----------------------------------------------------------------------------- public objective: six scales, per-scale upstream
def _weighted(losses, scales, coef):
    c_total, c_s = coef
    obj = 0.0
    if c_total is not None:
        obj = obj + c_total * losses["loss"]
    for s, c in zip(scales, c_s):
        if c:
            obj = obj + c * losses["loss/%d" % s]
    return obj


def _oracle_weighted(pb, coef, want_T, dtype):
    cast = lambda t: t.detach().to(dtype)
    d = {s: cast(pb.disp[s]).requires_grad_(True) for s in pb.scales}
    T = {k: cast(v).requires_grad_(want_T and k != "s") for k, v in pb.T.items()}
    opts = OP.default_opts(scales=list(pb.scales))
    _, losses = OP.photometric_objective({k: cast(v) for k, v in pb.color.items()}, d, cast(pb.K), cast(pb.inv_K), T,
                                         pb.frame_ids, {k: cast(v) for k, v in pb.noise.items()}, opts)
    _weighted(losses, pb.scales, coef).backward()
    # (a scale whose loss carries no weight gets no gradient: zero, which the device must produce exactly)
    grads = {s: d[s].grad if d[s].grad is not None else torch.zeros_like(d[s]) for s in pb.scales}
    return {k: v.detach() for k, v in losses.items()}, grads, \
        {k: v.grad for k, v in T.items() if v.requires_grad}


# (frame_ids, (B, H, W), scales, ops.MULTISOURCE, pose gradients, (coefficient of loss, coefficients of loss/s))
UPSTREAM_CASES = [
    ("six scales", (0, "s"), (2, 64, 128), (0, 1, 2, 3, 4, 5), True, False, (0.8, (1.3, -0.4, 2.1, 0.25, 0.6, -1.1))),
    ("photo_ms", (0, "s"), (2, 64, 96), (0, 1, 2, 3), True, False, (0.7, (1.3, -0.4, 2.1, 0.25))),
    ("photo_mf", (0, -1, 1), (2, 64, 96), (0, 1, 2, 3), True, True, (0.7, (1.3, -0.4, 2.1, 0.25))),
    ("general kernel", (0, -1, 1), (2, 64, 96), (0, 1, 2, 3), False, True, (0.7, (1.3, -0.4, 2.1, 0.25))),
    ("loss/2 alone", (0, "s"), (2, 64, 96), (0, 1, 2, 3), True, False, (None, (0.0, 0.0, 1.0, 0.0))),
    ("loss/1 alone, photo_mf", (0, -1, 1), (2, 64, 96), (0, 1, 2, 3), True, True, (None, (0.0, 1.0, 0.0, 0.0))),
]


@pytest.mark.parametrize("name,frame_ids,shape,scales,multisource,want_T,coef", UPSTREAM_CASES,
                         ids=[c[0] for c in UPSTREAM_CASES])
def test_objective_per_scale_upstream_vs_oracle(lib, name, frame_ids, shape, scales, multisource, want_T, coef):
    """Backward of c * loss + sum_s c_s * loss/s with distinct c_s (the per-scale upstream scalars reach
    dmh_disp_grad's g_scale and the pose-gradient contraction), and six scales (per-scale photometric kernels and the
    generic transposed up-sampling at R = 16 and 32), against the fp32 oracle with the fp64 arbiter."""
    from depthmodelhardening_b200 import objective, ops
    B, H, W = shape
    pb = synth.photo_batch(batch=B, height=H, width=W, frame_ids=frame_ids, scales=scales, seed=131)
    ref, rgd, rgT = _oracle_weighted(pb, coef, want_T, torch.float32)
    _, rgd64, rgT64 = _oracle_weighted(pb, coef, want_T, torch.float64)
    g = pb.to(DEV)
    old = ops.MULTISOURCE
    ops.MULTISOURCE = multisource
    try:
        disps = {s: g.disp[s].clone().requires_grad_(True) for s in g.scales}
        Ts = {k: v.clone().requires_grad_(want_T and k != "s") for k, v in g.T.items()}
        losses, _ = objective.photometric_losses(g.color, disps, g.K, g.inv_K, Ts, g.frame_ids, g.scales, H, W,
                                                 noise=g.noise)
        _weighted(losses, g.scales, coef).backward()
        torch.cuda.synchronize()
    finally:
        ops.MULTISOURCE = old
    assert_close(losses["loss"], ref["loss"], TOL, "loss")
    for s in g.scales:
        assert_close(losses["loss/%d" % s], ref["loss/%d" % s], TOL, "loss/%d" % s)
        assert_grad_close(disps[s].grad, rgd[s], rgd64[s], TOL, "%s grad_disp_%d" % (name, s))
    for k, t in rgT.items():
        assert_grad_close(Ts[k].grad, t, rgT64[k], 1e-4, "%s grad_T %s" % (name, k), outlier_frac=0.0, slack=3.0)


def test_single_row_objective_is_refused(lib):
    """H = 1 has no vertical smoothness edge and no SSIM reflection row: the objective refuses it (the identity-loss
    and smoothness kernels need two rows) instead of computing a value, so the IEEE-division builds are reached only
    through a capture (below)."""
    from depthmodelhardening_b200 import objective
    pb = synth.photo_batch(batch=1, height=1, width=64, frame_ids=(0, "s"), scales=(0,), seed=3).to(DEV)
    with pytest.raises(RuntimeError, match="bad shape"):
        objective.photometric_losses(pb.color, pb.disp, pb.K, pb.inv_K, pb.T, pb.frame_ids, pb.scales, 1, 64,
                                     noise=pb.noise)


# ----------------------------------------------------------------------------- IEEE-division builds (first size in a capture)
# W - 1 of each case is a constant no other test verifies (dmh_const_div_exact caches per constant; W - 1 is checked
# first, so an unverified W - 1 alone selects the IEEE build)
CAPTURE_CASES = [
    ("photo_ms", (0, "s"), (1, 32, 4104), True, True, r"photo_ms_kernel<false>", r"photo_ms_kernel<true>"),
    ("photo_mf", (0, -1, 1), (1, 32, 4108), True, True, r"photo_mf_kernel<false, true>", r"photo_mf_kernel<true, true>"),
    ("photo_fast", (0, "s"), (1, 32, 4112), True, False, r"photo_fast_kernel<\w+, false,",
     r"photo_fast_kernel<\w+, true,"),
]


def _kernel_names(fn):
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, {e.name for e in prof.events()}


@pytest.mark.parametrize("name,frame_ids,shape,multisource,multiscale,ieee,fast", CAPTURE_CASES,
                         ids=[c[0] for c in CAPTURE_CASES])
def test_capture_at_first_seen_size_runs_ieee_build(lib, name, frame_ids, shape, multisource, multiscale, ieee, fast):
    """Forward + backward of the objective captured by a bare torch.cuda.graph at a size the process has not seen:
    the division constant cannot be verified inside the capture, so the graph holds the IEEE-division build.  Its
    replay must give the same bits as a later eager run (which takes the verified 3-instruction division) and agree
    with the oracle; the profiler shows which build each ran."""
    from depthmodelhardening_b200 import objective, ops
    B, H, W = shape
    pb = synth.photo_batch(batch=B, height=H, width=W, frame_ids=frame_ids, seed=171)
    g = pb.to(DEV)
    want_T = any(f != "s" for f in frame_ids[1:])
    disps = {s: g.disp[s].clone().requires_grad_(True) for s in g.scales}
    Ts = {k: v.clone().requires_grad_(want_T and k != "s") for k, v in g.T.items()}
    inputs = [disps[s] for s in g.scales] + [Ts[k] for k in Ts if Ts[k].requires_grad]

    def run():
        losses, _ = objective.photometric_losses(g.color, disps, g.K, g.inv_K, Ts, g.frame_ids, g.scales, H, W,
                                                 noise=g.noise)
        grads = torch.autograd.grad(losses["loss"], inputs)
        return [losses["loss"]] + [losses["loss/%d" % s] for s in g.scales] + list(grads)

    old = ops.MULTISOURCE, ops.MULTISCALE
    ops.MULTISOURCE, ops.MULTISCALE = multisource, multiscale
    try:
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            captured = run()
        _, replay_names = _kernel_names(graph.replay)
        assert lib.dmh_const_div_exact(W - 1) == 1
        eager, eager_names = _kernel_names(run)
    finally:
        ops.MULTISOURCE, ops.MULTISCALE = old
    assert any(re.search(ieee, n) for n in replay_names), "replay kernels: %s" % sorted(replay_names)
    assert not any(re.search(fast, n) for n in replay_names)
    assert any(re.search(fast, n) for n in eager_names), "eager kernels: %s" % sorted(eager_names)
    for i, (a, b) in enumerate(zip(captured, eager)):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32)), "output %d: replay and eager bits differ" % i
    # and both agree with the oracle (as in the whole-objective tests, up to 0.5 % knife-edge pixels: at 32 x 4104 the
    # coarse scales' fp32 oracle itself has that many elements beyond twice its typical error)
    ref, rgd, rgT = _oracle_weighted(pb, (1.0, (0.0,) * len(pb.scales)), want_T, torch.float32)
    _, rgd64, rgT64 = _oracle_weighted(pb, (1.0, (0.0,) * len(pb.scales)), want_T, torch.float64)
    assert_close(eager[0], ref["loss"], TOL, "loss")
    S = len(pb.scales)
    for i, s in enumerate(pb.scales):
        assert_close(eager[1 + i], ref["loss/%d" % s], TOL, "loss/%d" % s)
        assert_grad_close(eager[1 + S + i], rgd[s], rgd64[s], TOL, "%s grad_disp_%d" % (name, s), outlier_frac=5e-3)
    for j, k in enumerate([k for k in Ts if Ts[k].requires_grad]):
        assert_grad_close(eager[1 + 2 * S + j], rgT[k], rgT64[k], 1e-4, "%s grad_T %s" % (name, k), outlier_frac=0.0,
                          slack=3.0)
