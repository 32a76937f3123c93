"""GPU parity of the stage-1 patch kernels over the placements, masks and patch sizes the attacks actually use.

The attack classes place the patch 5-30 m away (`dist_range=range(5, 31, 2)`, `np.linspace(5, 30, ...)` for the
arbitrary-angle attack).  At 29 m the 260 x 300 patch covers about 45 x 39 canvas pixels: the warp shrinks it ~6.7
times, so the bilinear taps of neighbouring canvas pixels land on texels far apart and an error in canvas coordinates
grows ~6.7 times in patch coordinates.  Real object masks reach the patch border (a car whose wheels touch the bottom
edge), where the tap-validity logic of `patch_taps` and the zero padding decide the result; the ellipse mask of
`synth.patch_batch` is 0 there.  Every comparison runs against the fp32 oracle (`oracle/patch.py`) with the fp64 run
of the same code as arbiter, plus a check of the gradient's support that a max-relative error cannot see.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from depthmodelhardening_b200 import synth
from oracle import patch as OQ
from oracle.refload import CALIB_P2, write_calib
from tests.util import assert_close, assert_close_arb, assert_grad_close, rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-5
P34 = np.array(CALIB_P2, dtype=np.float64).reshape(3, 4)

# the attack classes' distances, plus the non-integer ones of Phy_obj_atk_arbi's np.linspace(5, 30, ...)
Z_GRID = sorted(set(float(z) for z in range(5, 31, 2)) | set(np.linspace(5, 30, 7).tolist()))
ALPHAS = [float(a) for a in range(-30, 31, 5)]
# angles off the 5-degree grid: two per distance, so that the grid as a whole visits all of them
ODD_ALPHAS = [float(a) for a in range(-30, 31, 2) if a % 5]
MASKS = ["ellipse", "ones", "silhouette"]
BATCH = len(ALPHAS) + 2


def silhouette(h, w):
    """The ellipse, a full-width band over the bottom rows and a column band on the left: a mask that reaches three
    edges of the patch, like a car whose wheels touch the bottom.  The bands' inner edges carry fractional values
    k/255, as anti-aliased PNG masks do."""
    m = synth.ellipse_mask(h, w)[0, 0].clone()
    nb, nc = max(1, h // 8), max(1, w // 10)
    m[h - nb:, :] = 1.0
    m[:, :nc] = 1.0

    def ramp(n, seed):
        return torch.tensor([((37 * i + seed) % 254 + 1) / 255.0 for i in range(n)], dtype=torch.float32)
    if h - nb - 1 >= 0 and nc < w:
        m[h - nb - 1, nc:] = torch.maximum(m[h - nb - 1, nc:], ramp(w - nc, 3))
    if nc < w and h - nb > 0:
        m[:h - nb, nc] = torch.maximum(m[:h - nb, nc], ramp(h - nb, 11))
    return m.view(1, 1, h, w).contiguous()


def make_mask(kind, h=synth.PATCH_H, w=synth.PATCH_W):
    if kind == "ellipse":
        return synth.ellipse_mask(h, w)
    if kind == "ones":
        return torch.ones(1, 1, h, w)
    return silhouette(h, w)


def grid_alphas(i):
    """Angles of the i-th distance of Z_GRID: the 5-degree grid plus two odd angles."""
    return ALPHAS + [ODD_ALPHAS[(2 * i) % len(ODD_ALPHAS)], ODD_ALPHAS[(2 * i + 1) % len(ODD_ALPHAS)]]


@pytest.fixture(scope="module")
def dev():
    from depthmodelhardening_b200 import _lib
    _lib.load()
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def calib(tmp_path_factory):
    return write_calib(str(tmp_path_factory.mktemp("calib")))


@pytest.fixture(scope="module")
def inputs():
    """Scenes and upstream gradient of one BATCH-item batch (CPU), and a patch per patch size."""
    scenes = synth.smooth_field((BATCH, 3, synth.ORI_H, synth.ORI_W), 1800)
    up = synth.randn((BATCH, 3, synth.SCENE_H, synth.SCENE_W), 1900) * 1e-3
    return scenes, up


def assert_grad_support(g, g64, what):
    """Every texel the fp64 gradient gives weight (|g64| > 1e-3 max) is non-zero in the kernel result, and every
    non-zero texel of the kernel result lies within one texel of the fp64 support: dropped or misplaced taps."""
    g, g64 = g.detach().cpu().double(), g64.detach().cpu().double()
    strong = g64.abs() > 1e-3 * float(g64.abs().max())
    missing = int((strong & (g == 0)).sum())
    near = F.max_pool2d((g64 != 0).double().view(-1, 1, *g64.shape[-2:]), 3, 1, 1).view(g64.shape) > 0
    stray = int(((g != 0) & ~near).sum())
    assert missing == 0 and stray == 0, "%s: %d texels of the fp64 support missing, %d written outside it" % (
        what, missing, stray)


def check_apply(dev, obj, mask, scenes, up, z0s, alphas, what, size=(320, 1024)):
    """apply_patch (autograd) and apply_patch_fwd_bwd against the fp32 oracle, arbitrated by fp64: adv scenes,
    resized masks, per-item mask sums, the patch gradient and its support.  Returns the fp64 gradient."""
    from depthmodelhardening_b200 import patch_ops
    ph, pw = obj.shape[-2:]
    o32 = obj.clone().requires_grad_(True)
    adv32, m32 = OQ.apply_patch(o32, mask, scenes, z0s, alphas, P34, size=size)
    (adv32 * up).sum().backward()
    o64 = obj.double().requires_grad_(True)
    adv64, m64 = OQ.apply_patch(o64, mask.double(), scenes.double(), z0s, alphas, P34, size=size)
    (adv64 * up.double()).sum().backward()
    place = patch_ops.homographies(z0s, alphas, P34, obj_hw=(ph, pw)).to(dev)
    obj_d, mask_d, scenes_d, up_d = obj.to(dev).requires_grad_(True), mask.to(dev), scenes.to(dev), up.to(dev)
    adv, m = patch_ops.apply_patch(obj_d, mask_d, scenes_d, place, size=size)
    (adv * up_d).sum().backward()
    assert_close_arb(adv, adv32, adv64, TOL, "adv scene " + what)
    assert_close_arb(m, m32, m64, TOL, "resized mask " + what)
    # per-item mask sums: 1e-6, or twice the fp32 oracle's own error against fp64 where that is larger -- rounding
    # of the fp32 sampling coordinates at the silhouette's hard and fractional edges moves its sums by up to 2e-6
    # beyond 15 m (measured on the oracle), and a kernel computes those coordinates in fp32 too
    s64 = m64.sum((1, 2, 3))
    assert_close(m.double().sum((1, 2, 3)), s64, max(1e-6, 2.0 * rel_err(m32.double().sum((1, 2, 3)), s64)),
                 "resized mask sums " + what)
    assert_grad_close(obj_d.grad, o32.grad, o64.grad, TOL, "grad patch " + what)
    assert_grad_support(obj_d.grad, o64.grad, "grad patch " + what)
    adv2, m2, gp2 = patch_ops.apply_patch_fwd_bwd(obj.to(dev), mask_d, scenes_d, place, up_d, size=size)
    assert torch.equal(adv2, adv) and torch.equal(m2, m)
    assert_grad_close(gp2, o32.grad, o64.grad, TOL, "grad patch (fast path) " + what)
    assert_grad_support(gp2, o64.grad, "grad patch (fast path) " + what)
    return o64.grad


# ----------------------------------------------------------------------------- A. placement grid
@pytest.mark.parametrize("mask_kind", MASKS)
@pytest.mark.parametrize("z0", Z_GRID)
def test_fused_patch_apply_placement_grid(dev, inputs, z0, mask_kind):
    """One batch per distance (so that the gradient's scale is alike within it), every angle of the grid."""
    scenes, up = inputs
    i = Z_GRID.index(z0)
    obj = synth.rand((1, 3, synth.PATCH_H, synth.PATCH_W), 1700 + i)
    mask = make_mask(mask_kind)
    g64 = check_apply(dev, obj, mask, scenes, up, [z0] * BATCH, grid_alphas(i), "z0=%g %s" % (z0, mask_kind))
    if mask_kind != "ellipse":
        # the batch really exercises the border: the patch's last row (clipped by the canvas at 5 m) or its first
        # column carries gradient
        assert (g64[..., -1, :] != 0).any() or (g64[..., :, 0] != 0).any()


def test_physical_trans_project_all_placements(dev, calib):
    """PhysicalTrans.project(is_all=True) over the attack classes' distances: 13 x 13 = 169 items in one
    dmh_perspective_fwd launch, against the oracle's per-item warps; the dmh_perspective_bwd gradient to the patch
    per distance."""
    from depthmodelhardening_b200.physical import PhysicalTrans
    obj = synth.rand((1, 3, synth.PATCH_H, synth.PATCH_W), 1710)
    mask = silhouette(synth.PATCH_H, synth.PATCH_W)
    dists = list(range(5, 31, 2))
    pt = PhysicalTrans(obj.to(dev).requires_grad_(True), mask.to(dev), {"path": calib}, (1, 3, 375, 1242),
                       dist_range=dists)
    imgs, masks, zs, als = pt.project(is_all=True)
    n = len(ALPHAS)
    assert imgs.shape == (len(dists) * n, 3, 375, 1242) and masks.shape == (len(dists) * n, 1, 375, 1242)
    assert zs == [z for z in dists for _ in ALPHAS] and als == ALPHAS * len(dists)
    up = synth.randn((n, 3, 375, 1242), 1910) * 1e-3
    for k, z in enumerate(dists):
        sl = slice(k * n, (k + 1) * n)
        o32, o64 = obj.clone().requires_grad_(True), obj.double().requires_grad_(True)
        i32, m32, _ = OQ.project_patch(o32, mask, zs[sl], als[sl], P34)
        i64, m64, _ = OQ.project_patch(o64, mask.double(), zs[sl], als[sl], P34)
        assert_close_arb(imgs[sl], i32, i64, TOL, "warped patch z0=%d" % z)
        assert_close_arb(masks[sl], m32, m64, TOL, "warped mask z0=%d" % z)
        (i32 * up).sum().backward()
        (i64 * up.double()).sum().backward()
        pt.obj_img.grad = None
        im_z, _, _, _ = pt.project(batch_size=n, z0_sample=[z] * n, alpha_sample=ALPHAS)
        (im_z * up.to(dev)).sum().backward()
        assert_grad_close(pt.obj_img.grad, o32.grad, o64.grad, TOL, "perspective bwd z0=%d" % z)
        assert_grad_support(pt.obj_img.grad, o64.grad, "perspective bwd z0=%d" % z)


# ----------------------------------------------------------------------------- B. bbox hint, mixed batches
def test_bbox_hint_and_mixed_batch(dev, inputs):
    """The Placement's bounding box is only a hint: with it and with the bare coefficients the forward is the same
    bits and the gradient the same up to the order of the fp32 atomics.  A batch mixing near and far items (the
    backward grid is sized by its largest box) equals one launch per item."""
    from depthmodelhardening_b200 import patch_ops
    scenes, up = inputs
    z0, al = [5.0, 29.0, 17.0, 9.0, 30.0], [-30.0, 25.0, 0.0, 14.0, -8.0]
    b = len(z0)
    obj = synth.rand((1, 3, synth.PATCH_H, synth.PATCH_W), 1720).to(dev)
    mask = silhouette(synth.PATCH_H, synth.PATCH_W).to(dev)
    sc, u = scenes[:b].to(dev), up[:b].to(dev)
    place = patch_ops.homographies(z0, al, P34).to(dev)
    adv, m, g = patch_ops.apply_patch_fwd_bwd(obj, mask, sc, place, u)
    g = g.clone()
    adv_c, m_c, g_c = patch_ops.apply_patch_fwd_bwd(obj, mask, sc, place.coeffs, u)
    assert torch.equal(adv, adv_c) and torch.equal(m, m_c)
    assert_close(g_c, g, 1e-6, "grad patch, bare coefficients vs Placement")
    g_sum = torch.zeros_like(g)
    for i in range(b):
        p_i = patch_ops.homographies(z0[i:i + 1], al[i:i + 1], P34).to(dev)
        adv_i, m_i, g_i = patch_ops.apply_patch_fwd_bwd(obj, mask, sc[i:i + 1], p_i, u[i:i + 1])
        assert torch.equal(adv_i, adv[i:i + 1]) and torch.equal(m_i, m[i:i + 1]), "item %d" % i
        g_sum += g_i
    assert_close(g, g_sum, 1e-6, "grad patch, mixed batch vs sum of per-item launches")


# ----------------------------------------------------------------------------- D. span table and table-free kernels
def test_span_table_and_table_free_kernels_agree(dev, inputs):
    """The 3-tap forward / backward kernels read their resize weights from a span table built on the first eager call
    for a size; a first call during CUDA-graph capture runs the table-free instantiations instead.  Both give the
    same forward bits and the same gradient up to the order of the fp32 atomics."""
    from depthmodelhardening_b200 import _lib, patch_ops
    from tests.test_gpu_patch import resize_regime
    size = (317, 1013)                       # used by no other test: its span table does not exist yet
    assert resize_regime((375, 1242), size) == "3-tap 84x24"
    lib = _lib.load()
    scenes, up = inputs
    z0, al = [5.0, 17.0, 29.0], [-30.0, 0.0, 25.0]
    obj = synth.rand((1, 3, synth.PATCH_H, synth.PATCH_W), 1730).to(dev)
    mask = silhouette(synth.PATCH_H, synth.PATCH_W).to(dev)
    sc = scenes[:3].to(dev)
    u = synth.randn((3, 3) + size, 1920).to(dev) * 1e-3
    place = patch_ops.homographies(z0, al, P34).to(dev)
    patch_ops.apply_patch_fwd_bwd(obj, mask, sc, place, up[:3].to(dev))      # warm-up at the default size
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        adv_g, m_g, g_g = patch_ops.apply_patch_fwd_bwd(obj, mask, sc, place, u, size=size)
    graph.replay()
    torch.cuda.synchronize()
    n0 = lib.dmh_launch_count()
    adv_e, m_e, g_e = patch_ops.apply_patch_fwd_bwd(obj, mask, sc, place, u, size=size)
    torch.cuda.synchronize()
    assert lib.dmh_launch_count() - n0 == 3, "forward, backward and the span-table build (the size was unseen)"
    n0 = lib.dmh_launch_count()
    patch_ops.apply_patch_fwd_bwd(obj, mask, sc, place, u, size=size)
    assert lib.dmh_launch_count() - n0 == 2
    assert torch.equal(adv_g, adv_e) and torch.equal(m_g, m_e)
    assert float(m_e.sum()) > 1000
    assert_close(g_g, g_e, 1e-6, "grad patch, table-free vs span table")


# ----------------------------------------------------------------------------- E. patch sizes, write guard
@pytest.mark.parametrize("mask_kind", ["ones", "silhouette"])
@pytest.mark.parametrize("obj_hw", [(259, 301), (31, 47), (2, 300), (375, 1242)])
def test_patch_sizes(dev, calib, inputs, obj_hw, mask_kind):
    """Odd, small, thin and canvas-sized patches (l_pad = (1242 - pw) // 2 rounds down for odd widths; the
    canvas-sized patch has no padding at all): the perspective warp through PhysicalTrans, the fused apply through
    patch_ops.homographies(obj_hw=...), and a gradient buffer longer than the patch whose tail stays zero."""
    from depthmodelhardening_b200 import patch_ops
    from depthmodelhardening_b200.physical import PhysicalTrans
    scenes, up = inputs
    h, w = obj_hw
    z0, al = [5.0, Z_GRID[3], 17.0, 29.0], [-30.0, 14.0, 0.0, 28.0]
    b = len(z0)
    obj = synth.rand((1, 3, h, w), 1740 + h)
    mask = make_mask(mask_kind, h, w)
    what = "%dx%d %s" % (h, w, mask_kind)
    # perspective warp (PhysicalTrans passes the patch's own size to the placement)
    pt = PhysicalTrans(obj.to(dev).requires_grad_(True), mask.to(dev), {"path": calib}, (1, 3, 375, 1242))
    imgs, masks, _, _ = pt.project(batch_size=b, z0_sample=z0, alpha_sample=al)
    o32, o64 = obj.clone().requires_grad_(True), obj.double().requires_grad_(True)
    i32, m32, _ = OQ.project_patch(o32, mask, z0, al, P34)
    i64, m64, _ = OQ.project_patch(o64, mask.double(), z0, al, P34)
    assert_close_arb(imgs, i32, i64, TOL, "warped patch " + what)
    assert_close_arb(masks, m32, m64, TOL, "warped mask " + what)
    upc = synth.randn((b, 3, 375, 1242), 1930) * 1e-3
    (i32 * upc).sum().backward()
    (i64 * upc.double()).sum().backward()
    (imgs * upc.to(dev)).sum().backward()
    assert_grad_close(pt.obj_img.grad, o32.grad, o64.grad, TOL, "perspective bwd " + what)
    assert_grad_support(pt.obj_img.grad, o64.grad, "perspective bwd " + what)
    # fused apply
    check_apply(dev, obj, mask, scenes[:b], up[:b], z0, al, what)
    # the scatter stays inside the patch: a longer gradient buffer keeps its tail at zero
    place = patch_ops.homographies(z0, al, P34, obj_hw=obj_hw).to(dev)
    n = 3 * h * w
    buf = torch.full((n + w + 8,), 7.0, device=dev)
    _, _, gp = patch_ops.apply_patch_fwd_bwd(obj.to(dev), mask.to(dev), scenes[:b].to(dev), place, up[:b].to(dev),
                                             grad_out=buf)
    assert gp.data_ptr() == buf.data_ptr()
    assert torch.count_nonzero(buf[n:]) == 0, "patch gradient written past the patch"
    _, _, gp_ref = patch_ops.apply_patch_fwd_bwd(obj.to(dev), mask.to(dev), scenes[:b].to(dev), place, up[:b].to(dev))
    assert_close(gp, gp_ref, 1e-6, "grad patch into a caller's buffer " + what)
