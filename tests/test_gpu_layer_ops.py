"""Op-level kernels behind the `layers` drop-ins and `ops` (csrc/photometric_ops.cu, csrc/warp_smooth.cu) against
float64, at the tile, reflection, broadcast and launch-limit edges where kernels go wrong, with the gradient of every
input; and the shape checks the wrappers make before any launch (CPU).

References:
  * the oracle's own functions (oracle/photometric.py) run on the device in float32 and float64; for grid_sample and
    the up-sampling, torch on the same device (the reference runs ATen on CUDA), with float64 as the arbiter;
  * the linear ops (backproject forward and backward, project3d forward, disp_to_depth, up-sampling forward and
    backward) also element by element against float64 within k * 2^-24 * sum|terms| (as in test_gpu_objective_glue):
    a dropped or duplicated term fails there even where the max-relative check passes;
  * where floor() of a sampling coordinate is involved (the grid gradient of grid_sample, the disparity gradient of
    the warp) an element may differ only at a pixel whose float64 sampling coordinate lies within a few float32 ulp of
    an integer, where float32 and float64 can pick different tap pairs; every other element is compared with no
    outliers allowed.
"""
import pytest
import torch
import torch.nn.functional as F

from depthmodelhardening_b200 import synth
from oracle import photometric as OP
from tests.util import _record, assert_close, assert_close_arb, assert_grad_close, assert_within, up_weights

U = 2.0 ** -24
TOL = 1e-5
DEV = "cuda:0"
F32, F64 = torch.float32, torch.float64
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    from depthmodelhardening_b200 import _lib
    _lib.load()     # fails loudly if the extension is missing
    return torch.device(DEV)


def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def _rand(shape, seed, lo=0.0, hi=1.0):
    return lo + (hi - lo) * torch.rand(shape, generator=_gen(seed), device=DEV)


def _randn(shape, seed):
    return torch.randn(shape, generator=_gen(seed), device=DEV)


def _grads(fn, inputs, up, dtype, req=None):
    """Output of fn(*leaves) and the gradients of sum(output * up) w.r.t. the leaves marked in `req` (all by
    default); every leaf is a fresh copy of an input in `dtype`."""
    req = req or [True] * len(inputs)
    xs = [x.detach().to(dtype).requires_grad_(r) for x, r in zip(inputs, req)]
    out = fn(*xs)
    gs = torch.autograd.grad((out * up.to(out.dtype)).sum(), [x for x, r in zip(xs, req) if r])
    return out.detach(), gs


def _near_integer(c, ulps):
    """float64 sampling coordinates within `ulps` float32 ulp of an integer: floor() may pick either tap pair."""
    _, e = torch.frexp(c)
    return (c - torch.round(c)).abs() <= ulps * torch.exp2((e - 24).to(c.dtype))


def _unnormalise(g, size, align_corners):
    return (g + 1) / 2 * (size - 1) if align_corners else ((g + 1) * size - 1) / 2


def _camera(B, H, W, seed, kb=None):
    """K, inv_K of the KITTI intrinsics with a small perturbation of inv_K's 3x3 block (every entry nonzero), and a
    random motion T; kb matrices each (B when None)."""
    kb = kb or B
    K, inv_K = synth.intrinsics(H, W, kb)
    inv_K = inv_K.to(DEV)
    inv_K[:, :3, :3] += 1e-3 * _randn((kb, 3, 3), seed)
    T = synth.temporal_T(kb, seed + 1).to(DEV)
    T[:, :3, 3] *= 4.0
    return K.to(DEV), inv_K, T


# ----------------------------------------------------------------------------- case tables
# (B, C, H, W)
SSIM_CASES = [
    (2, 3, 2, 2), (1, 1, 3, 3), (2, 3, 2, 3), (2, 16, 3, 2),
    (2, 3, 16, 32), (1, 3, 17, 33), (2, 1, 16, 33), (1, 16, 17, 32),
    (21845, 3, 2, 2),
    (2, 3, 320, 1024),
]
# (B, C, H, W), each run with no_ssim False and True
REPROJ_CASES = [
    (2, 3, 2, 2), (1, 1, 3, 3), (2, 3, 3, 2),
    (2, 3, 16, 32), (1, 3, 17, 33), (2, 1, 17, 32),
    (21845, 3, 2, 2),
    (2, 3, 320, 1024),
]
# (B, C, h, w), each run with normalise False (get_smooth_loss) and True
SMOOTH_CASES = [(1, 3, 2, 40), (12, 1, 40, 2), (2, 8, 48, 80), (12, 3, 24, 80), (1, 3, 192, 640), (2, 1, 130, 130)]
# (B, H, W, batch of inv_K)
BACKPROJECT_CASES = [(2, 12, 21, 2), (3, 17, 33, 3), (96, 6, 20, 1), (2, 48, 80, 2)]
# (B, H, W, batch of K and T)
PROJECT_CASES = [(2, 10, 20, 2), (3, 17, 33, 3), (4, 24, 40, 1), (2, 48, 80, 2)]
# (B, H, W)
DISP_CASES = [(2, 10, 30), (2, 400, 800)]
# (B, C, Hs, Ws, Ho, Wo, grid kind)
GRID_CASES = [
    (2, 1, 9, 13, 7, 11, "random"),
    (2, 5, 20, 28, 17, 23, "random"),
    (1, 16, 33, 40, 31, 50, "random"),
    (2, 3, 5, 5, 14, 14, "special"),
    (1, 5, 8, 8, 14, 14, "special"),
]
# grid values of the "special" kind, every (x, y) pair of them: -1 / 1 are the borders with align_corners=True,
# -7/8 and 7/8 those of an 8-pixel axis with align_corners=False, W = 5 puts -1, -1/2, 0, 1/2, 1 on integer pixels
# with align_corners=True; then beyond the border, beyond the int range, and non-finite
SPECIAL = [-1.0, -0.875, -0.5, 0.0, 0.5, 0.875, 1.0, -1.5, 1.5, 1e10, -1e10, float("nan"), float("inf"),
           float("-inf")]
# (B, C, H, W, input_is_depth, batch of T)
WARP_CASES = [(2, 3, 24, 40, False, 2), (2, 1, 24, 33, False, 2), (2, 4, 20, 33, True, 1), (1, 3, 9, 33, True, 1)]
# (planes, h, w, H, W)
UPSAMPLE_CASES = [(2, 6, 10, 24, 40), (3, 40, 64, 17, 23), (2, 1, 10, 8, 40), (2, 12, 1, 24, 5), (2, 10, 16, 35, 24)]


def _ssim_regimes(B, C, H, W):
    r = {"C=%d" % C}
    r |= {"%s=%d" % (a, n) for a, n in (("H", H), ("W", W)) if n in (2, 3)}
    if W % 32 == 0:
        r.add("W=32k")                  # exact tile columns (32 x 16 tiles)
    if W > 32 and W % 32 == 1:
        r.add("W=32k+1")                # one extra column
    if H % 16 == 0:
        r.add("H=16k")
    if H > 16 and H % 16 == 1:
        r.add("H=16k+1")
    if B * C == 65535:
        r.add("B*C=65535")              # the grid-z limit
    if (H, W) == (320, 1024):
        r.add("320x1024")
    return r


def _smooth_regimes(B, C, h, w):
    r = {"C=%d" % C, "B=%d" % B, "hw<64*256" if h * w < 64 * 256 else "hw>64*256"}
    r |= {"%s=2" % a for a, n in (("h", h), ("w", w)) if n == 2}
    if h * w > 256:
        r.add("several loss blocks")
    return r


def _pixels_regimes(B, H, W, kb):
    N = H * W
    r = {"N<256" if N < 256 else ("N%256!=0" if N % 256 else "N%256==0")}
    if kb == 1 and B > 1:
        r.add("(1,4,4)")
    if B == 96 and kb == 1:
        r.add("B=96 (1,4,4)")
    return r


def _warp_regimes(B, C, H, W, isd, tb):
    r = {"C=%d" % C}
    if isd:
        r.add("depth input")
    if W == 33:
        r.add("W=33")
    if (H * W) % 256:
        r.add("N%256!=0")
    if tb == 1:
        r.add("T (1,4,4)")
    return r


def _upsample_regimes(P, h, w, H, W):
    r = set()
    if H < h or W < w:
        r.add("down")
    if h == 1 or w == 1:
        r.add("h or w = 1")
    if H * w != W * h:
        r.add("H/h != W/w")
    return r


def test_case_tables_reach_every_regime():
    def union(f, cases):
        return set().union(*(f(*c) for c in cases))
    assert union(_ssim_regimes, SSIM_CASES) >= {"H=2", "H=3", "W=2", "W=3", "W=32k", "W=32k+1", "H=16k", "H=16k+1",
                                                "C=1", "C=3", "C=16", "B*C=65535", "320x1024"}
    assert union(_ssim_regimes, REPROJ_CASES) >= {"H=2", "H=3", "W=2", "W=3", "W=32k", "W=32k+1", "H=16k", "H=16k+1",
                                                  "C=1", "C=3", "B*C=65535", "320x1024"}
    assert union(_smooth_regimes, SMOOTH_CASES) >= {"C=1", "C=3", "C=8", "h=2", "w=2", "hw<64*256", "hw>64*256",
                                                    "several loss blocks", "B=1", "B=12"}
    assert union(_pixels_regimes, BACKPROJECT_CASES) >= {"N<256", "N%256!=0", "B=96 (1,4,4)"}
    assert union(_pixels_regimes, PROJECT_CASES) >= {"N<256", "N%256!=0", "(1,4,4)"}
    assert max(B * H * W for B, H, W in DISP_CASES) > 148 * 16 * 256          # dmh_disp_to_depth's grid-stride loop
    assert {c[1] for c in GRID_CASES} >= {1, 5, 16} and {c[-1] for c in GRID_CASES} == {"random", "special"}
    assert any(c[4] * c[5] != c[2] * c[3] for c in GRID_CASES)
    assert {(c[2], c[3]) for c in GRID_CASES if c[-1] == "special"} >= {(5, 5), (8, 8)}
    assert union(_warp_regimes, WARP_CASES) >= {"C=1", "C=3", "C=4", "depth input", "W=33", "N%256!=0", "T (1,4,4)"}
    assert union(_upsample_regimes, UPSAMPLE_CASES) >= {"down", "h or w = 1", "H/h != W/w"}


# ----------------------------------------------------------------------------- SSIM / reprojection loss
@gpu
@pytest.mark.parametrize("B,C,H,W", SSIM_CASES)
def test_ssim_vs_fp64(dev, B, C, H, W):
    from depthmodelhardening_b200 import layers as L
    seed = B + 7 * C + 31 * H + 101 * W
    xy = [_rand((B, C, H, W), seed), _rand((B, C, H, W), seed + 1)]
    up = _randn((B, C, H, W), seed + 2)
    out, g = _grads(L.SSIM(), xy, up, F32)
    r32, g32 = _grads(OP.ssim, xy, up, F32)
    r64, g64 = _grads(OP.ssim, xy, up, F64)
    what = "ssim %dx%dx%dx%d" % (B, C, H, W)
    assert_close_arb(out, r32, r64, TOL, what)
    assert_grad_close(g[0], g32[0], g64[0], TOL, what + " grad_x", outlier_frac=0)
    assert_grad_close(g[1], g32[1], g64[1], TOL, what + " grad_y", outlier_frac=0)


@gpu
@pytest.mark.parametrize("no_ssim", [False, True])
@pytest.mark.parametrize("B,C,H,W", REPROJ_CASES)
def test_reprojection_loss_vs_fp64(dev, B, C, H, W, no_ssim):
    from depthmodelhardening_b200 import ops
    seed = 3 + B + 7 * C + 31 * H + 101 * W
    pt = [_rand((B, C, H, W), seed), _rand((B, C, H, W), seed + 1)]
    up = _randn((B, 1, H, W), seed + 2)
    out, g = _grads(lambda p, t: ops.reprojection_loss(p, t, no_ssim), pt, up, F32)
    r32, g32 = _grads(lambda p, t: OP.reprojection_loss(p, t, no_ssim), pt, up, F32)
    r64, g64 = _grads(lambda p, t: OP.reprojection_loss(p, t, no_ssim), pt, up, F64)
    what = "reproj %dx%dx%dx%d no_ssim=%d" % (B, C, H, W, no_ssim)
    assert_close_arb(out, r32, r64, TOL, what)
    assert_grad_close(g[0], g32[0], g64[0], TOL, what + " grad_pred", outlier_frac=0)
    assert_grad_close(g[1], g32[1], g64[1], TOL, what + " grad_target", outlier_frac=0)


@gpu
def test_ssim_grid_z_limit_is_refused(dev):
    """B*C = 65536 planes exceed the launch's grid z: refused on the host, nothing launched."""
    from depthmodelhardening_b200 import layers as L
    from depthmodelhardening_b200 import ops
    x = torch.rand(16384, 4, 2, 2, device=dev)
    with pytest.raises(RuntimeError, match="bad shape"):
        L.SSIM()(x, x)
    p = torch.rand(32768, 2, 2, 2, device=dev, requires_grad=True)
    loss = ops.reprojection_loss(p, torch.rand(32768, 2, 2, 2, device=dev))     # forward: grid z = B
    with pytest.raises(RuntimeError, match="bad shape"):
        loss.sum().backward()                                                    # backward: grid z = B*C


# ----------------------------------------------------------------------------- smoothness
@gpu
@pytest.mark.parametrize("normalise", [False, True])
@pytest.mark.parametrize("B,C,h,w", SMOOTH_CASES)
def test_smooth_loss_vs_fp64(dev, B, C, h, w, normalise):
    from depthmodelhardening_b200 import layers as L
    from depthmodelhardening_b200 import ops
    seed = 5 + B + 7 * C + 31 * h + 101 * w
    disp = 0.02 + 0.3 * _rand((B, 1, h, w), seed)
    img = _rand((B, C, h, w), seed + 1)
    up = torch.tensor(0.7, device=dev)
    fn = (lambda d, i: ops.smooth_loss(d, i, normalise=True)) if normalise else L.get_smooth_loss
    ref = OP.normalised_smooth_loss if normalise else OP.smooth_loss
    out, g = _grads(fn, [disp, img], up, F32)
    r32, g32 = _grads(ref, [disp, img], up, F32)
    r64, g64 = _grads(ref, [disp, img], up, F64)
    what = "smooth %dx%dx%dx%d normalise=%d" % (B, C, h, w, normalise)
    assert_close_arb(out, r32, r64, TOL, what)
    assert_grad_close(g[0], g32[0], g64[0], TOL, what + " grad_disp", outlier_frac=0)
    assert_grad_close(g[1], g32[1], g64[1], TOL, what + " grad_img", outlier_frac=0)


@gpu
def test_smooth_image_gradient_beyond_eight_channels_is_refused(dev):
    from depthmodelhardening_b200 import ops
    d = (0.1 + _rand((1, 1, 8, 8), 1)).requires_grad_(True)
    img = _rand((1, 9, 8, 8), 2).requires_grad_(True)
    loss = ops.smooth_loss(d, img)
    with pytest.raises(RuntimeError, match="C <= 8"):
        loss.backward()


# ----------------------------------------------------------------------------- BackprojectDepth
@gpu
@pytest.mark.parametrize("B,H,W,kb", BACKPROJECT_CASES)
def test_backproject_vs_fp64(dev, B, H, W, kb):
    """Points, the depth gradient and the inv_K gradient (the 3x3 block; summed over the batch by the expand of a
    (1,4,4) matrix), every element within its rounding bound:
      points_i = d * (iK_i0 x + iK_i1 y + iK_i2): 4 roundings;
      grad_depth = sum_i g_i * ray_i: 3 per ray + 3;
      grad_inv_K_ij = sum_n g_i(n) d(n) pix_j(n): 2 per term, 8 in the block tree of 256, then the sums over the
      blocks and over the expanded batch (at most one rounding per summand)."""
    from depthmodelhardening_b200 import layers as L
    seed = B + 7 * H + 31 * W + kb
    _, inv_K, _ = _camera(B, H, W, seed, kb)
    depth = 1.0 / (0.01 + 9.99 * _rand((B, 1, H, W), seed + 3))
    N = H * W
    up = _randn((B, 4, N), seed + 4)
    bp = L.BackprojectDepth(B, H, W)
    pts, (gd, giK) = _grads(bp, [depth, inv_K], up, F32)
    r32, g32 = _grads(OP.backproject, [depth, inv_K], up, F32)
    r64, g64 = _grads(OP.backproject, [depth, inv_K], up, F64)
    what = "backproject B=%d %dx%d inv_K batch %d" % (B, H, W, kb)
    assert_close_arb(pts, r32, r64, TOL, what)
    assert_grad_close(gd, g32[0], g64[0], TOL, what + " grad_depth", outlier_frac=0)
    assert_grad_close(giK, g32[1], g64[1], TOL, what + " grad_inv_K", outlier_frac=0)
    # element-wise
    iK = inv_K.double()[:, :3, :3].expand(B, 3, 3)
    pix = OP.pixel_grid(B, H, W, DEV, F64)                                    # (B,3,N): x, y, 1
    d = depth.double().view(B, 1, N)
    terms = d.abs() * torch.matmul(iK.abs(), pix)
    assert_within(pts[:, :3], r64[:, :3], 4 * U * terms, what + " points")
    assert torch.equal(pts[:, 3], torch.ones_like(pts[:, 3]))
    g = up.double()[:, :3]
    ray_terms = torch.matmul(iK.abs(), pix)                                    # (B,3,N)
    assert_within(gd.view(B, N), g64[0].view(B, N), 6 * U * (g.abs() * ray_terms).sum(1), what + " grad_depth")
    nblk = -(-N // 256)
    gi_terms = torch.einsum("bin,bjn->bij", (g * d).abs(), pix)
    k = 10 + nblk + (B if kb == 1 else 0)
    if kb == 1:
        gi_terms = gi_terms.sum(0, keepdim=True)
    assert_within(giK[:, :3, :3], g64[1][:, :3, :3], k * U * gi_terms, what + " grad_inv_K")
    assert torch.equal(giK[:, 3], torch.zeros_like(giK[:, 3])) and torch.equal(giK[:, :, 3], torch.zeros_like(giK[:, :, 3]))


# ----------------------------------------------------------------------------- Project3D
@gpu
@pytest.mark.parametrize("B,H,W,kb", PROJECT_CASES)
def test_project3d_vs_fp64(dev, B, H, W, kb):
    """Grid, and the gradients of the points (the homogeneous row included), K and T.  The grid, element by element:
    P = K @ T and p = P @ pt take 4 roundings each (8 on p through P), z = p2 + eps one more, u = p0 / z, / (W-1),
    - 0.5 one each; so |d gx| <= 2 * [8u S0 / (|z| (W-1)) + |n| (8u S2 / |z| + 3u)] + 2u |n - 0.5| with
    S_i = sum_jk |K_ik T_kj pt_j| and n = u / (W-1) (likewise for gy)."""
    from depthmodelhardening_b200 import layers as L
    seed = 11 + B + 7 * H + 31 * W + kb
    K, inv_K, T = _camera(B, H, W, seed, kb)
    depth = 1.0 / (0.01 + 9.99 * _rand((B, 1, H, W), seed + 3))
    pts = OP.backproject(depth, inv_K.expand(B, 4, 4)).detach()
    up = _randn((B, H, W, 2), seed + 4)
    pj = L.Project3D(B, H, W)
    grid, g = _grads(pj, [pts, K, T], up, F32)
    fn = lambda p, k, t: OP.project3d(p, k, t, H, W)
    r32, g32 = _grads(fn, [pts, K, T], up, F32)
    r64, g64 = _grads(fn, [pts, K, T], up, F64)
    what = "project3d B=%d %dx%d K/T batch %d" % (B, H, W, kb)
    assert_close_arb(grid, r32, r64, TOL, what)
    for i, name in enumerate(("points", "K", "T")):
        assert_grad_close(g[i], g32[i], g64[i], TOL, what + " grad_" + name, outlier_frac=0)
    # element-wise
    Kd, Td, pd = K.double().expand(B, 4, 4), T.double().expand(B, 4, 4), pts.double()
    cam = torch.matmul(torch.matmul(Kd, Td)[:, :3], pd)                        # (B,3,N)
    S = torch.einsum("bik,bkj,bjn->bin", Kd.abs(), Td.abs(), pd.abs())[:, :3]
    z = (cam[:, 2] + 1e-7).abs()
    for a, size in ((0, W), (1, H)):
        n = cam[:, a] / (cam[:, 2] + 1e-7) / (size - 1)
        bound = 2 * (8 * U * S[:, a] / (z * (size - 1)) + n.abs() * (8 * U * S[:, 2] / z + 3 * U)) \
            + 2 * U * (n - 0.5).abs()
        assert_within(grid[..., a].reshape(B, -1), r64[..., a].reshape(B, -1), bound, what + " grid[%d]" % a)


# ----------------------------------------------------------------------------- disp_to_depth
@gpu
@pytest.mark.parametrize("B,H,W", DISP_CASES)
def test_disp_to_depth_vs_fp64(dev, B, H, W):
    """Both outputs in the loss.  scaled = min_disp + range * disp with the two constants rounded to float32: 3
    roundings on (min_disp + range |disp|); depth = 1 / scaled correctly rounded."""
    from depthmodelhardening_b200 import layers as L
    disp = _rand((B, 1, H, W), B + H + W)
    u1, u2 = _randn((B, 1, H, W), 1), _randn((B, 1, H, W), 2)
    mn, mx = 0.1, 100.0

    def run(fn, dtype):
        d = disp.to(dtype).requires_grad_(True)
        s, dp = fn(d, mn, mx)
        (g,) = torch.autograd.grad((s * u1.to(dtype)).sum() + (dp * u2.to(dtype)).sum(), [d])
        return s.detach(), dp.detach(), g

    s, dp, g = run(L.disp_to_depth, F32)
    s32, dp32, g32 = run(OP.disp_to_depth, F32)
    s64, dp64, g64 = run(OP.disp_to_depth, F64)
    what = "disp_to_depth %dx%dx%d" % (B, H, W)
    assert_close_arb(s, s32, s64, TOL, what + " scaled")
    assert_close_arb(dp, dp32, dp64, TOL, what + " depth")
    assert_grad_close(g, g32, g64, TOL, what + " grad", outlier_frac=0)
    terms = 1.0 / mx + (1.0 / mn - 1.0 / mx) * disp.double().abs()
    assert_within(s, s64, 3 * U * terms, what + " scaled")
    assert_within(dp, dp64, dp64.abs() * (3 * U * terms / s64.abs() + U), what + " depth")


# ----------------------------------------------------------------------------- grid_sample
def _special_grid(B, seed):
    v = torch.tensor(SPECIAL, dtype=F32)
    n = len(SPECIAL)
    g = torch.stack([v.view(1, n).expand(n, n), v.view(n, 1).expand(n, n)], -1)      # (n, n, 2): every (x, y)
    gs = [g.roll(b, 0) for b in range(B)]
    return torch.stack(gs).to(DEV).contiguous()


@gpu
@pytest.mark.parametrize("pad,ac", [("zeros", True), ("zeros", False), ("border", True), ("border", False)])
@pytest.mark.parametrize("B,C,Hs,Ws,Ho,Wo,kind", GRID_CASES)
def test_grid_sample_vs_torch_cuda(dev, B, C, Hs, Ws, Ho, Wo, kind, pad, ac):
    """Against ATen on the same device (fp64 arbiter).  Random grids: the grid gradient may differ only where the
    float64 sampling coordinate is within 4 ulp of an integer (ATen's align_corners=False unnormalisation may be
    contracted into an FMA).  Special grids (exact borders, exact integer pixels, beyond the int range, NaN, +-inf):
    coordinates are exact, so every element is compared; ATen's gradient is zero at a clipped border, and a NaN
    coordinate scatters nothing in its backward.  The special grids are compared with ATen's own CUDA kernel: with
    zeros padding and align_corners=True torch dispatches to cuDNN by default, which turns a NaN coordinate into a
    NaN sample where ATen's kernel (and this one) drop the sample."""
    from depthmodelhardening_b200 import ops
    seed = B + 7 * C + 31 * Hs + 101 * Ws + 3 * Ho + Wo + (pad == "border") + 2 * ac
    src = _rand((B, C, Hs, Ws), seed)
    grid = _rand((B, Ho, Wo, 2), seed + 1, -1.3, 1.3) if kind == "random" else _special_grid(B, seed)
    assert grid.shape == (B, Ho, Wo, 2)
    up = _randn((B, C, Ho, Wo), seed + 2)
    ref = lambda s, g: F.grid_sample(s, g, mode="bilinear", padding_mode=pad, align_corners=ac)
    out, (gs, gg) = _grads(lambda s, g: ops.grid_sample(s, g, padding_mode=pad, align_corners=ac), [src, grid], up, F32)
    with torch.backends.cudnn.flags(enabled=kind == "random"):
        r32, (gs32, gg32) = _grads(ref, [src, grid], up, F32)
        r64, (gs64, gg64) = _grads(ref, [src, grid], up, F64)
    what = "grid_sample %s %s ac=%d C=%d %dx%d->%dx%d" % (kind, pad, ac, C, Hs, Ws, Ho, Wo)
    for t in (out, gs, gg):
        assert torch.isfinite(t).all(), what
    assert_close_arb(out, r32, r64, TOL, what)
    assert_grad_close(gs, gs32, gs64, TOL, what + " grad_src", outlier_frac=0)
    if kind == "special":
        assert_grad_close(gg, gg32, gg64, TOL, what + " grad_grid", outlier_frac=0)
        return
    g64 = grid.double()
    near = _near_integer(_unnormalise(g64[..., 0], Ws, ac), 4) | _near_integer(_unnormalise(g64[..., 1], Hs, ac), 4)
    keep = (~near).unsqueeze(-1).expand_as(gg)
    _record("explained", what + " grad_grid", near_integer_pixels=int(near.sum()), pixels=near.numel())
    assert_grad_close(gg[keep], gg32[keep], gg64[keep], TOL, what + " grad_grid", outlier_frac=0)


# ----------------------------------------------------------------------------- fused warp
def _warp_oracle(isd, H, W):
    def fn(x, src, K, T, inv_K, ac=True):
        if isd:
            depth = x
        else:
            _, depth = OP.disp_to_depth(x, 0.1, 100.0)
        grid = OP.project3d(OP.backproject(depth, inv_K.expand(x.shape[0], 4, 4)), K, T, H, W)
        return F.grid_sample(src, grid, padding_mode="border", align_corners=ac), grid, depth
    return fn


def _warp_inputs(B, C, H, W, isd, tb, seed):
    K, inv_K, T = _camera(B, H, W, seed, tb)
    K = K[:1].expand(B, 4, 4).contiguous() if tb == 1 else K
    disp = 0.02 + 0.3 * _rand((B, 1, H, W), seed + 5)
    x = 1.0 / (0.01 + 9.99 * disp) if isd else disp
    return x, _rand((B, C, H, W), seed + 6), K, T, inv_K


@gpu
@pytest.mark.parametrize("B,C,H,W,isd,tb", WARP_CASES)
def test_warp_reproject_vs_fp64(dev, B, C, H, W, isd, tb):
    """warp_reproject against the oracle chain (disp_to_depth -> BackprojectDepth -> Project3D -> grid_sample(border,
    align_corners=True)): the warped image and the disparity (or depth), source, K and T gradients.  The disparity
    gradient may differ only where the float64 sampling coordinate is within 16 ulp of an integer (the float32 chain
    takes ~16 roundings)."""
    from depthmodelhardening_b200 import ops
    seed = 13 + B + 7 * C + 31 * H + 101 * W + isd + tb
    x, src, K, T, inv_K = _warp_inputs(B, C, H, W, isd, tb, seed)
    up = _randn((B, C, H, W), seed + 7)
    fn = lambda x_, s_, k_, t_: ops.warp_reproject(x_, s_, k_, inv_K, t_, 0.1, 100.0, input_is_depth=isd)
    orc = _warp_oracle(isd, H, W)
    out, g = _grads(fn, [x, src, K, T], up, F32)
    r32, g32 = _grads(lambda *a: orc(*a, inv_K.float())[0], [x, src, K, T], up, F32)
    r64, g64 = _grads(lambda *a: orc(*a, inv_K.double())[0], [x, src, K, T], up, F64)
    what = "warp C=%d B=%d %dx%d depth=%d T batch %d" % (C, B, H, W, isd, tb)
    assert_close_arb(out, r32, r64, TOL, what)
    for i, name in ((1, "src"), (2, "K"), (3, "T")):
        assert_grad_close(g[i], g32[i], g64[i], TOL, what + " grad_" + name, outlier_frac=0)
    with torch.no_grad():
        _, grid64, _ = orc(x.double(), src.double(), K.double(), T.double(), inv_K.double())
    near = _near_integer(_unnormalise(grid64[..., 0], W, True), 16) | \
        _near_integer(_unnormalise(grid64[..., 1], H, True), 16)
    keep = ~near.unsqueeze(1)
    _record("explained", what + " grad_disp", near_integer_pixels=int(near.sum()), pixels=near.numel())
    assert_grad_close(g[0][keep], g32[0][keep], g64[0][keep], TOL, what + " grad_disp", outlier_frac=0)


@gpu
@pytest.mark.parametrize("ac", [True, False])
@pytest.mark.parametrize("isd", [False, True])
def test_warp_with_aux_vs_fp64(dev, ac, isd):
    """The no-grad warp with its sampling grid and depth; align_corners=False is the depth-hints warp."""
    from depthmodelhardening_b200 import ops
    B, C, H, W = 2, 3, 24, 33
    x, src, K, T, inv_K = _warp_inputs(B, C, H, W, isd, 2, 17 + ac + 2 * isd)
    orc = _warp_oracle(isd, H, W)
    with torch.no_grad():
        out = ops.warp_with_aux(x, src, K, inv_K, T, 0.1, 100.0, input_is_depth=isd, align_corners=ac)
        r32 = orc(x, src, K, T, inv_K, ac)
        r64 = orc(x.double(), src.double(), K.double(), T.double(), inv_K.double(), ac)
    for name, a, b, c in zip(("warped", "grid", "depth"), out, r32, r64):
        assert_close_arb(a, b, c, TOL, "warp_with_aux ac=%d depth=%d %s" % (ac, isd, name))


# ----------------------------------------------------------------------------- up-sampling
@gpu
@pytest.mark.parametrize("P,h,w,H,W", UPSAMPLE_CASES)
def test_upsample_bilinear_vs_fp64(dev, P, h, w, H, W):
    """Against F.interpolate on the same device (fp64 arbiter), and every element against float64 with the kernels'
    float32 interpolation weights: forward 5 roundings per tap (two products, two adds, the weight sum of a clamped
    tap), backward ntx + nty + 2 (row and column sums of the gather)."""
    from depthmodelhardening_b200 import ops
    seed = P + 7 * h + 31 * w + 3 * H + W
    x = _rand((P, 1, h, w), seed)
    up = _randn((P, 1, H, W), seed + 1)
    ref = lambda t: F.interpolate(t, [H, W], mode="bilinear", align_corners=False)
    out, (g,) = _grads(lambda t: ops.upsample_bilinear(t, (H, W)), [x], up, F32)
    r32, (g32,) = _grads(ref, [x], up, F32)
    r64, (g64,) = _grads(ref, [x], up, F64)
    what = "upsample %dx%d->%dx%d" % (h, w, H, W)
    assert_close_arb(out, r32, r64, TOL, what)
    assert_grad_close(g, g32, g64, TOL, what + " grad", outlier_frac=0)
    Ay = torch.from_numpy(up_weights(H, h)).to(DEV)
    Ax = torch.from_numpy(up_weights(W, w)).to(DEV)
    x64, G = x.double()[:, 0], up.double()[:, 0]
    fwd = torch.einsum("Yy,pyx,Xx->pYX", Ay, x64, Ax)
    fwd_abs = torch.einsum("Yy,pyx,Xx->pYX", Ay.abs(), x64.abs(), Ax.abs())
    assert_within(out[:, 0], fwd, 5 * U * fwd_abs, what + " forward")
    bwd = torch.einsum("Yy,pYX,Xx->pyx", Ay, G, Ax)
    bwd_abs = torch.einsum("Yy,pYX,Xx->pyx", Ay.abs(), G.abs(), Ax.abs())
    k = int((Ax != 0).sum(0).max()) + int((Ay != 0).sum(0).max()) + 2
    assert_within(g[:, 0], bwd, k * U * bwd_abs, what + " backward")


# ----------------------------------------------------------------------------- dtype, layout, determinism
def _specs():
    """name -> (inputs, fn, indices of the inputs whose gradient is an atomic (RED) scatter, needs grad)."""
    from depthmodelhardening_b200 import layers as L
    from depthmodelhardening_b200 import ops
    B, H, W = 2, 12, 21
    K, inv_K, T = _camera(B, H, W, 40)
    img = lambda s, c=3: _rand((B, c, H, W), s)
    disp = 0.02 + 0.3 * _rand((B, 1, H, W), 41)
    depth = 1.0 / (0.01 + 9.99 * disp)
    pts = OP.backproject(depth, inv_K).detach()
    grid = _rand((B, 9, 11, 2), 42, -1.2, 1.2)
    return {
        "ssim": ([img(1), img(2)], L.SSIM(), (), True),
        "reprojection_loss": ([img(3), img(4)], lambda p, t: ops.reprojection_loss(p, t), (), True),
        "reprojection_loss no_ssim": ([img(3), img(4)], lambda p, t: ops.reprojection_loss(p, t, True), (), True),
        "get_smooth_loss": ([disp, img(5)], L.get_smooth_loss, (), True),
        "smooth_loss normalised": ([disp, img(5)], lambda d, i: ops.smooth_loss(d, i, True), (), True),
        "BackprojectDepth": ([depth, inv_K], L.BackprojectDepth(B, H, W), (), True),
        "Project3D": ([pts, K, T], L.Project3D(B, H, W), (), True),
        "disp_to_depth": ([disp], lambda d: torch.cat(L.disp_to_depth(d, 0.1, 100.0), 1), (), True),
        "grid_sample border": ([img(6), grid], lambda s, g: ops.grid_sample(s, g, padding_mode="border",
                                                                             align_corners=True), (0,), True),
        "grid_sample zeros": ([img(6), grid], lambda s, g: ops.grid_sample(s, g, padding_mode="zeros"), (0,), True),
        "warp_reproject": ([disp, img(7), K, T], lambda d, s, k, t: ops.warp_reproject(d, s, k, inv_K, t), (1,), True),
        "warp_reproject C=4": ([disp, img(8, 4), K, T], lambda d, s, k, t: ops.warp_reproject(d, s, k, inv_K, t), (1,),
                               True),
        "warp_with_aux": ([depth, img(9), K, T],
                          lambda d, s, k, t: torch.cat([a.flatten() for a in ops.warp_with_aux(
                              d, s, k, inv_K, t, input_is_depth=True, align_corners=False)]), (), False),
        "upsample_bilinear": ([disp], lambda d: ops.upsample_bilinear(d, (17, 45)), (), True),
    }


SPEC_NAMES = ["ssim", "reprojection_loss", "reprojection_loss no_ssim", "get_smooth_loss", "smooth_loss normalised",
              "BackprojectDepth", "Project3D", "disp_to_depth", "grid_sample border", "grid_sample zeros",
              "warp_reproject", "warp_reproject C=4", "warp_with_aux", "upsample_bilinear"]


def _run_spec(fn, inputs, need_grad):
    if not need_grad:
        with torch.no_grad():
            return fn(*inputs), ()
    leaves = [x.detach().requires_grad_(True) for x in inputs]
    out = fn(*leaves)
    up = _randn(out.shape, 99)
    return out.detach(), torch.autograd.grad((out.float() * up).sum(), leaves)


def _non_contiguous(x):
    """A channels_last copy of an image with several channels, else every other element of a twice-as-wide buffer."""
    if x.dim() == 4 and x.shape[1] > 1:
        return x.contiguous(memory_format=torch.channels_last)
    buf = torch.empty(*x.shape[:-1], 2 * x.shape[-1], device=x.device, dtype=x.dtype)
    v = buf[..., ::2]
    v.copy_(x)
    return v


@gpu
@pytest.mark.parametrize("name", SPEC_NAMES)
def test_bf16_non_contiguous_and_repeat(dev, name):
    """bf16 inputs give the float32 result of the widened values, and their gradients come back in bf16; a
    non-contiguous input gives what the contiguous one gives; a second run gives the same bits (atomic scatters of a
    source-image gradient excepted, which are compared within 1e-5)."""
    inputs, fn, atomic, need_grad = _specs()[name]
    assert sorted(SPEC_NAMES) == sorted(_specs())
    out, g = _run_spec(fn, inputs, need_grad)
    out2, g2 = _run_spec(fn, inputs, need_grad)
    assert out.dtype == F32 and torch.equal(out, out2), name + ": output differs between two runs"
    for i, (a, b) in enumerate(zip(g, g2)):
        if i in atomic:
            assert_close(a, b, TOL, name + " grad %d, second run" % i)
        else:
            assert torch.equal(a, b), name + ": gradient %d differs between two runs" % i
    # bf16
    xb = [x.to(torch.bfloat16) for x in inputs]
    ob, gb = _run_spec(fn, xb, need_grad)
    ow, gw = _run_spec(fn, [x.float() for x in xb], need_grad)
    assert ob.dtype == F32 and torch.equal(ob, ow), name + ": bf16 output != output of the widened input"
    for i, (a, b) in enumerate(zip(gb, gw)):
        assert a.dtype == torch.bfloat16, name + ": gradient %d comes back as %s" % (i, a.dtype)
        if i in atomic:
            assert_close(a.float(), b.to(torch.bfloat16).float(), 2.0 ** -7, name + " bf16 grad %d" % i)
        else:
            assert torch.equal(a, b.to(torch.bfloat16)), name + ": bf16 gradient %d" % i
    # non-contiguous
    xn = [_non_contiguous(x) for x in inputs]
    assert not any(x.is_contiguous() for x in xn)
    on, gn = _run_spec(fn, xn, need_grad)
    assert torch.equal(on, out), name + ": non-contiguous input changes the output"
    for i, (a, b) in enumerate(zip(gn, g)):
        if i in atomic:
            assert_close(a, b, TOL, name + " non-contiguous grad %d" % i)
        else:
            assert torch.equal(a, b), name + ": non-contiguous input changes gradient %d" % i


# ----------------------------------------------------------------------------- host-side contract (CPU)
def _cpu_camera():
    K, inv_K = synth.intrinsics(8, 8, 2)
    return K, inv_K, synth.stereo_T(2)


SHAPE_MISMATCHES = {
    "grid_sample batch": (lambda L, ops: ops.grid_sample(torch.rand(2, 3, 8, 8), torch.rand(3, 4, 4, 2)),
                          "same batch size"),
    "grid_sample last dim": (lambda L, ops: ops.grid_sample(torch.rand(2, 3, 8, 8), torch.rand(2, 4, 4, 3)),
                             "size 2 in last dimension"),
    "SSIM": (lambda L, ops: L.SSIM()(torch.rand(2, 3, 8, 8), torch.rand(2, 3, 8, 9)), "same shape"),
    "reprojection_loss": (lambda L, ops: ops.reprojection_loss(torch.rand(2, 3, 8, 8), torch.rand(2, 1, 8, 8)),
                          "same shape"),
    "get_smooth_loss size": (lambda L, ops: L.get_smooth_loss(torch.rand(2, 1, 8, 8), torch.rand(2, 3, 8, 9)),
                             "matching img"),
    "smooth_loss batch": (lambda L, ops: ops.smooth_loss(torch.rand(3, 1, 8, 8), torch.rand(2, 3, 8, 8), True),
                          "matching img"),
    "smooth_loss disp channels": (lambda L, ops: L.get_smooth_loss(torch.rand(2, 3, 8, 8), torch.rand(2, 3, 8, 8)),
                                  "matching img"),
    "warp_reproject": (lambda L, ops: ops.warp_reproject(torch.rand(2, 1, 8, 9), torch.rand(2, 3, 8, 8),
                                                         *_cpu_camera()[:2], _cpu_camera()[2]), "matching src"),
    "warp_with_aux": (lambda L, ops: ops.warp_with_aux(torch.rand(1, 1, 8, 8), torch.rand(2, 3, 8, 8),
                                                       *_cpu_camera()), "matching src"),
    "Project3D": (lambda L, ops: L.Project3D(2, 8, 8)(torch.rand(2, 3, 64), *_cpu_camera()[::2]), r"\(B,4,N\)"),
}


@pytest.mark.parametrize("name", sorted(SHAPE_MISMATCHES))
def test_shape_mismatch_raises_before_launch(name):
    """CPU tensors: the shape check comes first, so the shape error (not the CUDA-only one) is raised."""
    from depthmodelhardening_b200 import layers as L
    from depthmodelhardening_b200 import ops
    call, words = SHAPE_MISMATCHES[name]
    with pytest.raises(RuntimeError, match=words):
        call(L, ops)


def test_fused_warps_refuse_gradients_they_do_not_return():
    from depthmodelhardening_b200 import ops
    K, inv_K, T = _cpu_camera()
    d, src = torch.rand(2, 1, 8, 8), torch.rand(2, 3, 8, 8)
    with pytest.raises(RuntimeError, match="no gradient w.r.t. inv_K"):
        ops.warp_reproject(d, src, K, inv_K.clone().requires_grad_(True), T)
    with pytest.raises(RuntimeError, match="returns no gradient"):
        ops.warp_with_aux(d.requires_grad_(True), src, K, inv_K, T)
    with torch.no_grad(), pytest.raises(RuntimeError, match="CUDA-only"):
        ops.warp_reproject(d, src, K, inv_K.clone().requires_grad_(True), T)
