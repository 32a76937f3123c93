"""GPU parity: stage-1 CUDA kernels (through the C ABI / ctypes) against the
oracle and the reference goldens.

Integer / index work is compared bit-exactly: projected corners (host), the L0
survivor set and count, the top-k selection, the L-inf update (pure clamp/sign
arithmetic).  Floating point: <= 1e-5 relative on warped patches, composited
scenes and patch gradients (atomics make the gradient's summation order
run-dependent, still within tolerance).
"""
import random

import numpy as np
import pytest
import torch

from depthmodelhardening_b200 import synth
from oracle import patch as OQ
from oracle.refload import CALIB_P2, write_calib
from tests.util import assert_close, assert_close_arb, load_golden, rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-5
P34 = np.array(CALIB_P2, dtype=np.float64).reshape(3, 4)


@pytest.fixture(scope="module")
def dev():
    from depthmodelhardening_b200 import _lib
    _lib.load()
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def calib(tmp_path_factory):
    return write_calib(str(tmp_path_factory.mktemp("calib")))


def crop(t):
    return t[..., 100:228, 440:760]


def test_physical_trans_project_vs_golden(dev, calib):
    from depthmodelhardening_b200.physical import PhysicalTrans
    g = load_golden("patch")
    pbt = synth.patch_batch(batch=3, seed=0).to(dev)
    pt = PhysicalTrans(pbt.obj.clone().requires_grad_(True), pbt.mask, {"path": calib}, (1, 3, 375, 1242))
    z0, al = g["z0"].tolist(), g["alpha"].tolist()
    imgs, masks, zs, als = pt.project(batch_size=3, z0_sample=z0, alpha_sample=al)
    assert imgs.shape == (3, 3, 375, 1242) and masks.shape == (3, 1, 375, 1242) and zs == z0 and als == al
    assert_close(crop(imgs), g["proj_img_crop"], TOL, "proj img")
    assert_close(crop(masks), g["proj_mask_crop"], TOL, "proj mask")
    assert_close(imgs.double().sum(), g["proj_img_sum"], 1e-6)
    assert_close(masks.double().sum(), g["proj_mask_sum"], 1e-6)
    for i, (z, a) in enumerate(zip(z0, al)):
        assert np.array_equal(pt.objPosOnImage(z, a), g["corners"][i])
    K = np.array([[0.58 * 1242, 0, 0.5 * 1242, 0], [0, 1.92 * 375, 0.5 * 375, 0], [0, 0, 1, 0], [0, 0, 0, 1]],
                 dtype=np.float32)
    T = np.eye(4, dtype=np.float32)
    T[0, 3] = -0.1
    imgs_k, masks_k = pt.project_w_trans(T, z0, al, K=K)
    i64, _, _ = OQ.project_patch(pbt.obj.cpu().double(), pbt.mask.cpu().double(), z0, al, P34, K=K, T=T)
    assert_close_arb(crop(imgs_k), g["projk_img_crop"], crop(i64), TOL, "projk img")
    assert_close(masks_k.double().sum(), g["projk_mask_sum"], 1e-6)
    # reference composite + Resize on our warps, gradient to the patch through the perspective backward
    adv = OQ.resize_aa(pbt.scenes * (1 - masks) + imgs * masks)
    (adv * pbt.upstream).sum().backward()
    assert_close(adv[:, :, 90:200, 380:640], g["adv_crop"], TOL, "adv crop")
    assert_close(pt.obj_img.grad[:, :, ::3, ::3], g["grad_patch"], TOL, "grad patch (perspective bwd)")


@pytest.mark.parametrize("batch", [3, 8])
def test_fused_patch_apply_vs_oracle(dev, batch):
    from depthmodelhardening_b200 import patch_ops
    pbt = synth.patch_batch(batch=batch, seed=2)
    obj = pbt.obj.clone().requires_grad_(True)
    adv_ref, m_ref = OQ.apply_patch(obj, pbt.mask, pbt.scenes, pbt.z0, pbt.alpha, P34)
    (adv_ref * pbt.upstream).sum().backward()
    g = pbt.to(dev)
    co = patch_ops.homographies(pbt.z0, pbt.alpha, P34).to(dev)
    obj_d = g.obj.clone().requires_grad_(True)
    adv, m = patch_ops.apply_patch(obj_d, g.mask, g.scenes, co)
    (adv * g.upstream).sum().backward()
    o64 = pbt.obj.double().requires_grad_(True)
    adv64, m64 = OQ.apply_patch(o64, pbt.mask.double(), pbt.scenes.double(), pbt.z0, pbt.alpha, P34)
    (adv64 * pbt.upstream.double()).sum().backward()
    assert_close_arb(adv, adv_ref, adv64, TOL, "adv scene")
    assert_close_arb(m, m_ref, m64, TOL, "resized mask")
    assert_close_arb(obj_d.grad, obj.grad, o64.grad, TOL, "grad patch")
    # the no-autograd fast path gives the same three results
    adv2, m2, gp2 = patch_ops.apply_patch_fwd_bwd(g.obj, g.mask, g.scenes, co, g.upstream)
    assert torch.equal(adv2, adv) and torch.equal(m2, m)
    assert_close_arb(gp2, obj.grad, o64.grad, TOL, "grad patch (fast path)")


def resize_regime(in_hw, out_hw):
    """The forward kernel dmh_patch_apply_fwd selects for a resize, restated op by op in float32 (aa_tile_extent
    and the host selection of patch.cu): "3-tap 84x24" / "3-tap 104x30" (both scale factors < 1.5, tile extents
    within the compile-time tile), "generic 8-tap" (larger down-scales) or "refused" (a factor >= 3)."""
    f = np.float32
    sy, sx = f(in_hw[0]) / f(out_hw[0]), f(in_hw[1]) / f(out_hw[1])
    if sy >= 3 or sx >= 3:
        return "refused"

    def extent(tile, s):
        support = s if s >= 1 else f(1)
        return int(f(f(s * f(tile)) + f(f(2) * support)) + f(3))
    if sy < 1.5 and sx < 1.5:
        return "3-tap 84x24" if extent(64, sx) <= 84 and extent(16, sy) <= 24 else "3-tap 104x30"
    return "generic 8-tap"


def bwd_window_reach(in_size, out_size):
    """patch_apply_bwd_kernel visits, for one canvas pixel ci, the outputs ox_a(ci) + k; the first 8 (MAXO) from
    registers, the rest in its remainder loop.  Returns 1 + the largest k at which an output actually reads ci with a
    non-zero weight (3-tap spans, float32 as in the kernel): above 8 the remainder loop contributes."""
    f = np.float32
    s = f(in_size) / f(out_size)
    sup = s if s >= 1 else f(1)
    inv = f(1) / s if s >= 1 else f(1)
    o = np.arange(out_size)
    center = (s * (o.astype(np.float32) + f(0.5))).astype(np.float32)
    lo = np.maximum((center - sup + f(0.5)).astype(np.float32).astype(np.int64), 0)
    n = np.minimum(np.minimum((center + sup + f(0.5)).astype(np.float32).astype(np.int64), in_size) - lo, 3)
    reach = 0
    for j in range(3):
        arg = ((f(j) + (lo.astype(np.float32) - center)).astype(np.float32) + f(0.5)).astype(np.float32) * inv
        ci = lo + j
        live = (j < n) & (np.abs(arg) < 1)
        ox_a = np.maximum(0, np.floor(((ci.astype(np.float32) - sup).astype(np.float32) - f(0.5)) / s).astype(np.int64) - 1)
        if live.any():
            reach = max(reach, int((o - ox_a)[live].max()) + 1)
    return reach


# the resize regime each output size of 375 x 1242 is meant to exercise: a retuned switch point fails loudly
RAGGED_SIZES = {(321, 1030): "3-tap 84x24", (200, 650): "generic 8-tap", (375, 1242): "3-tap 84x24",
                (160, 512): "generic 8-tap", (270, 900): "3-tap 104x30",
                (307, 1000): "3-tap 84x24",        # top of the 84 x 24 tile (extents 84 / 24)
                (306, 999): "3-tap 104x30",        # just over it (85 / 25)
                (307, 999): "3-tap 104x30", (306, 1000): "3-tap 104x30",      # one axis over the limit each
                (251, 829): "3-tap 104x30",        # scales 1.494 / 1.498: the 8-row vertical window can be full
                (250, 828): "generic 8-tap",       # exactly 1.5
                (126, 415): "generic 8-tap",       # 2.98 / 2.99: the largest shared-memory tile
                (640, 2048): "3-tap 84x24", (750, 2484): "3-tap 84x24",      # up-scaling, within 8 outputs
                (960, 3200): "3-tap 84x24"}        # up-scaling by 2.56 / 2.58
# output sizes whose backward reads outputs beyond the 8 it keeps in registers (bwd_window_reach > 8)
REMAINDER_SIZES = {(960, 3200)}


@pytest.mark.parametrize("size", list(RAGGED_SIZES))
def test_fused_patch_apply_ragged_output_sizes(dev, size):
    """Output sizes that are not multiples of the 64 x 16 tile, on both sides of every switch between the resize
    kernels (3-tap windows in an 84 x 24 or a 104 x 30 tile, the generic 8-tap kernel), the identity resize and
    up-scales, one of them far enough that the backward reads outputs beyond the 8 it keeps in registers: forward
    and the gradient to the patch against the oracle, with the ellipse mask and with an all-ones mask that reaches
    the patch border."""
    from depthmodelhardening_b200 import patch_ops
    assert resize_regime((375, 1242), size) == RAGGED_SIZES[size]
    assert (bwd_window_reach(1242, size[1]) > 8) == (size in REMAINDER_SIZES)
    pbt = synth.patch_batch(batch=2, seed=3)
    up = synth.randn((2, 3) + size, 904) * 1e-3
    g = pbt.to(dev)
    co = patch_ops.homographies(pbt.z0, pbt.alpha, P34).to(dev)
    for kind, mask in (("ellipse", pbt.mask), ("ones", torch.ones_like(pbt.mask))):
        what = "%s %s" % (size, kind)
        obj = pbt.obj.clone().requires_grad_(True)
        adv_ref, m_ref = OQ.apply_patch(obj, mask, pbt.scenes, pbt.z0, pbt.alpha, P34, size=size)
        (adv_ref * up).sum().backward()
        o64 = pbt.obj.double().requires_grad_(True)
        adv64, m64 = OQ.apply_patch(o64, mask.double(), pbt.scenes.double(), pbt.z0, pbt.alpha, P34, size=size)
        (adv64 * up.double()).sum().backward()
        obj_d = g.obj.clone().requires_grad_(True)
        adv, m = patch_ops.apply_patch(obj_d, mask.to(dev), g.scenes, co, size=size)
        (adv * up.to(dev)).sum().backward()
        assert torch.isfinite(adv).all() and torch.isfinite(m).all()
        assert_close_arb(adv, adv_ref, adv64, TOL, "adv scene " + what)
        assert_close_arb(m, m_ref, m64, TOL, "resized mask " + what)
        assert_close_arb(obj_d.grad, obj.grad, o64.grad, TOL, "grad patch " + what)


@pytest.mark.parametrize("size", [(125, 414), (100, 400)])
def test_fused_patch_apply_refuses_down_scale_of_3(dev, size):
    """A down-scale factor of 3 or more needs anti-aliasing windows wider than the kernels' 8 taps: refused."""
    from depthmodelhardening_b200 import patch_ops
    assert resize_regime((375, 1242), size) == "refused"
    g = synth.patch_batch(batch=2, seed=3).to(dev)
    co = patch_ops.homographies(g.z0, g.alpha, P34).to(dev)
    up = torch.zeros((2, 3) + size, device=dev)
    with pytest.raises(RuntimeError, match="down-scale factor"):
        patch_ops.apply_patch(g.obj, g.mask, g.scenes, co, size=size)
    with pytest.raises(RuntimeError, match="down-scale factor"):
        patch_ops.apply_patch_fwd_bwd(g.obj, g.mask, g.scenes, co, up, size=size)


def test_fused_patch_apply_vs_golden(dev):
    from depthmodelhardening_b200 import patch_ops
    g = load_golden("patch")
    pbt = synth.patch_batch(batch=3, seed=0).to(dev)
    z0, al = g["z0"].tolist(), g["alpha"].tolist()
    co = patch_ops.homographies(z0, al, P34).to(dev)
    obj = pbt.obj.clone().requires_grad_(True)
    adv, m = patch_ops.apply_patch(obj, pbt.mask, pbt.scenes, co)
    (adv * pbt.upstream).sum().backward()
    assert_close(adv.reshape(-1)[torch.from_numpy(g["adv_idx"]).to(dev)], g["adv_samples"], TOL, "adv samples")
    assert_close(adv.double().sum(), g["adv_sum"], 1e-7)
    assert_close(adv[:, :, 90:200, 380:640], g["adv_crop"], TOL, "adv crop")
    assert_close(m[:, :, 90:200, 380:640], g["mask_rs_crop"], TOL, "mask crop")
    assert_close(m.double().sum(), g["mask_rs_sum"], 1e-6)
    assert_close(obj.grad[:, :, ::3, ::3], g["grad_patch"], TOL, "grad patch")
    assert_close(obj.grad.double().sum(), g["grad_patch_sum"], 1e-5)


def test_patch_apply_batch_mismatch_raises(dev):
    from depthmodelhardening_b200 import patch_ops
    pbt = synth.patch_batch(batch=2, seed=0).to(dev)
    co = patch_ops.homographies([5, 6, 7], [0, 5, 10], P34).to(dev)
    with pytest.raises(RuntimeError, match="Batch size"):
        patch_ops.apply_patch(pbt.obj, pbt.mask, pbt.scenes, co)


def test_pgd_linf_step_bit_exact(dev):
    from depthmodelhardening_b200 import patch_ops
    clean = synth.rand((1, 3, 260, 300), 1)
    adv = (clean + (synth.rand(clean.shape, 2) - 0.5) * 0.2).clamp(0, 1)
    grad = synth.randn(clean.shape, 3)
    grad[0, 0, :5, :5] = 0.0                      # sign(0) == 0
    ref = OQ.pgd_linf_step(adv, grad, clean, 0.02, 0.1)
    out = patch_ops.pgd_linf_step(adv.to(dev), grad.to(dev), clean.to(dev), 0.02, 0.1)
    assert torch.equal(out.cpu(), ref)


def test_l0_compose_count_and_finalize_bit_exact(dev):
    from depthmodelhardening_b200 import patch_ops
    obj = synth.rand((1, 3, 260, 300), 11)
    # patterns around the 1/255 threshold, some negative / above 1, exact cancellations included
    pp = (synth.rand(obj.shape, 12) - 0.3) * 0.02
    pn = (synth.rand(obj.shape, 13) - 0.3) * 0.02
    pp[0, :, 10:20, 10:20] = 0.5
    pn[0, :, 10:20, 10:20] = 0.5               # pos + neg cancels exactly -> not counted
    pp[0, :, 30:40, :] = 1.7
    adv_ref, pos, neg = OQ.l0_compose(obj, pp, pn)
    cnt_ref, surv_ref = OQ.l0_count(pos, neg)
    st = patch_ops.L0State(obj.to(dev), pp.to(dev), pn.to(dev))
    adv = st.compose_count(first=True)
    assert torch.equal(adv.cpu(), adv_ref)
    assert int(st.counts[0]) == int(cnt_ref) and int(st.counts[1]) == int(cnt_ref)
    assert int(patch_ops.l0_count(obj.to(dev), pp.to(dev), pn.to(dev))) == int(cnt_ref)
    fin_ref, fpos, fneg = OQ.l0_finalize(obj, pp, pn)
    fin, pattern = st.finalize()
    assert torch.equal(fin.cpu(), fin_ref)
    assert torch.equal(pattern.cpu(), fpos + fneg)
    surv = (pattern.abs().sum(1) != 0).cpu()
    assert torch.equal(surv, surv_ref)         # bit-exact L0 surviving-pixel set


def test_l0_adam_step_vs_torch_autograd(dev):
    """mask-cost gradient + clamp chain + Adam in one kernel vs autograd + torch.optim.Adam."""
    from depthmodelhardening_b200 import patch_ops
    obj = synth.rand((1, 3, 64, 80), 21)
    pp0, pn0 = synth.rand(obj.shape, 22) * 1.2 - 0.1, synth.rand(obj.shape, 23) * 1.2 - 0.1
    g_adv_steps = [synth.randn(obj.shape, 24 + i) * 1e-3 for i in range(3)]
    pp = pp0.clone().requires_grad_(True)
    pn = pn0.clone().requires_grad_(True)
    opt = torch.optim.Adam([pp, pn], lr=0.5, betas=(0.5, 0.9))
    st = patch_ops.L0State(obj.to(dev), pp0.to(dev), pn0.to(dev), lr=0.5)
    for i, g_adv in enumerate(g_adv_steps):
        mask_w = 0.06 if i != 1 else 0.0
        adv, pos, neg = OQ.l0_compose(obj, pp, pn)
        cost = (adv * g_adv).sum() + mask_w * OQ.l0_mask_cost(pp, pn)
        opt.zero_grad()
        cost.backward()
        opt.step()
        st.compose_count(first=(i == 0))
        st.counts[1] = 1 if i != 1 else 10 ** 9          # force ratio > / <= thresh on the device
        st.adam_step(g_adv.to(dev), 0.06, 0.1)
        assert_close(st.ppos, pp, 2e-6, "P+ after step %d" % i)
        assert_close(st.pneg, pn, 2e-6, "P- after step %d" % i)


def test_l0_attack_iteration_graph_replay_equals_eager(dev):
    """Adam's step index lives on the device (dmh_l0_adam_step_dev): (a) the device-step update equals the host-step
    one (dmh_l0_adam_step) bit for bit over several steps, through the point where the mask weight switches off;
    (b) ONE captured attack iteration (compose + count -> fused patch apply -> update with a fixed gradient), replayed n times,
    leaves the same patterns, moments and counts as n eager iterations -- a host-side step index would be frozen
    into the capture and mis-scale every replay after the first."""
    from depthmodelhardening_b200 import patch_ops
    from oracle.refload import CALIB_P2
    pt_cpu = synth.patch_batch(batch=2, seed=9)
    pt = pt_cpu.to(dev)
    P34 = np.array(CALIB_P2, dtype=np.float64).reshape(3, 4)
    coeffs = patch_ops.homographies(pt_cpu.z0, pt_cpu.alpha, P34, obj_hw=(synth.PATCH_H, synth.PATCH_W)).to(dev)

    def make(device_step):
        return patch_ops.L0State(pt.obj, pt.pattern_pos, pt.pattern_neg, lr=0.5, betas=(0.5, 0.9), device_step=device_step)

    # the patch gradient of the iteration: computed ONCE (the backward scatters with fp32 atomics -- its last bits
    # differ from launch to launch) and fed to every instance
    adv0 = make(False).compose_count(first=True)
    _, _, grad0 = patch_ops.apply_patch_fwd_bwd(adv0, pt.mask, pt.scenes, coeffs, pt.upstream)
    grad0 = grad0.clone()

    def iteration(st, first=False):
        adv = st.compose_count(first=first)
        patch_ops.apply_patch(adv, pt.mask, pt.scenes, coeffs)       # (the forward placement: deterministic)
        st.adam_step(grad0, 0.06, 0.1)

    def state(st):
        return [t.clone() for t in (st.ppos, st.pneg, st.m_pos, st.v_pos, st.m_neg, st.v_neg, st.counts)]

    n = 6
    host, devs = make(False), make(True)
    for i in range(n):
        iteration(host, first=(i == 0))
        iteration(devs, first=(i == 0))
        for a, b in zip(state(host), state(devs)):
            assert torch.equal(a, b), "device-step vs host-step after iteration %d" % i
    assert int(devs.step_state[0]) == n and int(devs.step_state[1]) == 0
    # (b) graph replay
    g = make(True)
    iteration(g, first=True)                               # the init count is taken outside the capture
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph):
            iteration(g)
    torch.cuda.current_stream().wait_stream(side)
    # (capturing does not execute: the state is still the one after the first eager iteration)
    for _ in range(n - 1):
        graph.replay()
    torch.cuda.synchronize()
    for a, b in zip(state(host), state(g)):
        assert torch.equal(a, b), "graph replay vs eager"
    assert int(g.step_state[0]) == n


@pytest.mark.parametrize("k", [0, 1, 777, 40000, 78000, 90000])
def test_topk_radix_select_bit_exact(dev, k):
    from depthmodelhardening_b200 import patch_ops
    pp = synth.rand((1, 3, 260, 300), 31) * 1.3 - 0.2
    pn = synth.rand((1, 3, 260, 300), 32) * 1.3 - 0.2
    # heavy ties: quantise a region, and a block of exact duplicates of the likely k-th value
    pp[0, :, :100] = torch.round(pp[0, :, :100] * 8) / 8
    pn[0, :, :100] = torch.round(pn[0, :, :100] * 8) / 8
    rp, rn, keep_ref = OQ.topk_l0_project(pp, pn, k)
    op, on, keep = patch_ops.topk_l0_project(pp.to(dev), pn.to(dev), k)
    assert torch.equal(keep.cpu(), keep_ref)   # bit-exact top-k selection incl. tie order
    assert torch.equal(op.cpu(), rp) and torch.equal(on.cpu(), rn)
    assert int(keep.sum()) == min(max(k, 0), 78000)


def _tiny(dev):
    """The stand-in depth network (outside the graft).  Its cuDNN convolutions are pinned to deterministic fp32:
    with TF32 / heuristic algorithm choice the network gradient carries ~1e-3 of noise that depends on the
    allocator state left by EARLIER tests (workspace size steers cuDNN's choice) -- the attack-loop comparisons
    below count sign flips at |grad| ~ 0 and were order-dependent because of it."""
    from oracle.make_golden import TinyDepth
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.deterministic = True
    torch.backends.cudnn.benchmark = False
    return TinyDepth().to(dev)


def test_linf_attack_class_vs_reference_golden(dev, calib):
    import os
    from depthmodelhardening_b200 import attacks
    g = load_golden("attack_linf")
    attacks.object_dataset_root = os.path.dirname(os.path.dirname(os.path.dirname(calib)))
    pbt = synth.patch_batch(batch=3, seed=0).to(dev)
    random.seed(5)
    atk = attacks.Phy_obj_atk(_tiny(dev), pbt.obj.clone(), pbt.mask.clone(), eps=0.1, alpha=0.02, steps=2,
                              random_start=False, dist_range=list(range(5, 10, 2)))
    adv_s, ben_s, m_out, obj_adv = atk(pbt.scenes.clone(), 3)
    assert adv_s.shape == (3, 3, 320, 1024) and m_out.shape == (3, 1, 320, 1024) and obj_adv.shape == (1, 3, 260, 300)
    # same placements (RNG order) -> masks / benign scenes match to fp32 tolerance
    assert_close(m_out.double().sum(), g["mask_out_sum"], 1e-6)
    assert_close(ben_s.double().sum(), g["ben_scene_sum"], 1e-6)
    # sign(grad) flips where |grad| ~ 0 (cuDNN vs CPU convolution rounding): bound the fraction
    diff = (obj_adv.cpu()[:, :, ::2, ::2] - torch.from_numpy(g["obj_adv"])).abs()
    assert float((diff > 1e-6).float().mean()) < 0.02
    assert_close(adv_s.double().sum(), g["adv_scene_sum"], 1e-4)
    with pytest.raises(RuntimeError, match="Batch size"):
        atk(pbt.scenes[:2].clone(), 3)


def test_pgd_l2_step_vs_oracle(dev):
    """dmh_pgd_l2_step (phy_obj_atk_l2.py:108-120 in one launch): inside the ball (no projection), outside it
    (projection + clamp) and the zero-gradient / zero-delta corner (eps / 0 -> factor 1)."""
    from depthmodelhardening_b200 import patch_ops
    clean = synth.rand((1, 3, 260, 300), 1)
    grad = synth.randn(clean.shape, 3) * 1e-4
    for adv, alpha, eps in ((clean.clone(), 0.5, 3.0), ((clean + 0.05 * synth.randn(clean.shape, 4)).clamp(0, 1), 2.5, 3.0),
                            (clean.clone(), 0.0, 1.0)):
        ref = OQ.pgd_l2_step(adv, grad, clean, alpha, eps)
        ref64 = OQ.pgd_l2_step(adv.double(), grad.double(), clean.double(), alpha, eps)
        out = patch_ops.pgd_l2_step(adv.to(dev), grad.to(dev), clean.to(dev), alpha, eps)
        assert_close_arb(out, ref, ref64, 1e-6, "l2 step alpha=%g" % alpha)
        assert float((out.cpu() - clean).double().norm()) <= eps * (1 + 1e-6)
    zero = patch_ops.pgd_l2_step(clean.to(dev), torch.zeros_like(clean).to(dev), clean.to(dev), 0.5, 1.0)
    assert torch.equal(zero.cpu(), clean)                       # 0 / (0 + 1e-10) = 0; eps / 0 = inf -> factor 1


@pytest.mark.parametrize("ev", [False, True])
def test_l2_attack_class_vs_reference_golden(dev, calib, ev):
    """Drop-in `Phy_obj_atk_l2` (next-4) against the unmodified reference class at batch size 1
    (oracle/make_golden_l2.py): same placements, patch within fp32 tolerance (no sign() in this update, so no
    knife-edge flips), scenes / masks to fp32 tolerance."""
    import os
    from depthmodelhardening_b200 import attacks
    g = load_golden("attack_l2")
    tag = "eval" if ev else "rand"
    attacks.object_dataset_root = os.path.dirname(os.path.dirname(os.path.dirname(calib)))
    pbt = synth.patch_batch(batch=1, seed=0).to(dev)
    random.seed(21)
    atk = attacks.Phy_obj_atk_l2(_tiny(dev), pbt.obj.clone(), pbt.mask.clone(), eps=3.0, steps=3, random_start=False,
                                 dist_range=list(range(5, 10, 2)))
    assert atk.alpha == 2.5 * 3.0 / 3
    adv_s, ben_s, m_out, obj_adv = atk(pbt.scenes.clone(), 1, eval=ev)
    assert adv_s.shape == (1, 3, 320, 1024) and m_out.shape == (1, 1, 320, 1024) and obj_adv.shape == (1, 3, 260, 300)
    assert_close(m_out.double().sum(), g[tag + "_mask_sum"], 1e-6)
    assert_close(ben_s.double().sum(), g[tag + "_ben_sum"], 1e-6)
    assert_close(obj_adv[:, :, ::2, ::2], g[tag + "_obj_adv"], 2e-4, "patch")      # cuDNN vs CPU convolution gradients
    assert_close((obj_adv - pbt.obj).double().norm(), g[tag + "_delta_norm"], 1e-5)
    assert_close(adv_s[:, :, 90:200:2, 380:640:2], g[tag + "_adv_crop"], 2e-4, "adv crop")
    with pytest.raises(RuntimeError, match="Batch size"):
        atk(pbt.scenes.repeat(2, 1, 1, 1), 3)
    # random start (device RNG) stays inside the ball and in [0,1]
    atk2 = attacks.Phy_obj_atk_l2(_tiny(dev), pbt.obj.clone(), pbt.mask.clone(), eps=0.5, steps=1, random_start=True,
                                  dist_range=list(range(5, 10, 2)))
    _, _, _, adv2 = atk2(pbt.scenes.clone(), 1)
    assert float((adv2 - pbt.obj).norm()) <= 0.5 * (1 + 1e-5) and float(adv2.min()) >= 0 and float(adv2.max()) <= 1


def test_l0_attack_class_vs_reference_golden(dev, calib):
    import os
    from depthmodelhardening_b200 import attacks
    g = load_golden("attack_l0")
    attacks.object_dataset_root = os.path.dirname(os.path.dirname(os.path.dirname(calib)))
    pbt = synth.patch_batch(batch=3, seed=0).to(dev)
    random.seed(6)
    np.random.seed(7)
    atk = attacks.Phy_obj_atk_l0(_tiny(dev), pbt.obj.clone(), pbt.mask.clone(), adam_lr=0.5, steps=2, mask_wt=0.06,
                                 l0_thresh=0.1, dist_range=list(range(5, 10, 2)))
    adv_s, ben_s, m_out, obj_adv = atk(pbt.scenes.clone(), 3)
    l0 = int(atk.cal_l0())
    assert abs(l0 - int(g["l0_count"])) <= 0.01 * int(g["l0_count"])
    surv = (atk.pattern.abs().sum(1) != 0).cpu().numpy().astype(np.uint8)
    surv_ref = np.unpackbits(g["survivors"])[:surv.size].reshape(surv.shape)
    assert np.mean(surv != surv_ref) < 0.01
    # Adam's first steps are sign-like (+-lr): elements whose tiny gradient changes sign between the CPU
    # reference run and this GPU run (cuDNN vs CPU convolution rounding) move by ~1; bound their fraction
    d = (atk.pattern_pos_tensor.cpu()[:, :, ::2, ::2] - torch.from_numpy(g["pattern_pos_tensor"])).abs()
    assert float((d > 1e-3).float().mean()) < 0.10
    assert_close(adv_s.double().sum(), g["adv_scene_sum"], 1e-3)


def _placements(seed, steps, ranges, batch):
    """The (z0, alpha) draws the attack classes make, in their RNG order."""
    random.seed(seed)
    out = []
    for _ in range(steps + 1):
        z0 = random.sample(ranges[0], batch)
        al = random.sample(ranges[1], batch)
        out.append((z0, al))
    return out[:-1], out[-1]


class _Monodepth2ResNet18(torch.nn.Module):
    """north_star's network shape: a random-init ResNet-18 encoder (torchvision) and monodepth2's depth decoder
    (reflection-padded 3x3 conv + ELU blocks, nearest x2 upsampling with skip connections, channels 16..256),
    returning the sigmoid disparity at full resolution."""

    def __init__(self):
        import torchvision
        super().__init__()
        nn = torch.nn
        self.enc = torchvision.models.resnet18(weights=None)
        ch_enc, ch_dec = [64, 64, 128, 256, 512], [16, 32, 64, 128, 256]

        def block(cin, cout):
            return nn.Sequential(nn.ReflectionPad2d(1), nn.Conv2d(cin, cout, 3), nn.ELU(inplace=True))
        self.up0 = nn.ModuleList(block(ch_enc[-1] if i == 4 else ch_dec[i + 1], ch_dec[i]) for i in range(5))
        self.up1 = nn.ModuleList(block(ch_dec[i] + (ch_enc[i - 1] if i > 0 else 0), ch_dec[i]) for i in range(5))
        self.disp = nn.Sequential(nn.ReflectionPad2d(1), nn.Conv2d(ch_dec[0], 1, 3))

    def forward(self, x):
        e = self.enc
        f = [e.relu(e.bn1(e.conv1((x - 0.45) / 0.225)))]
        f.append(e.layer1(e.maxpool(f[0])))
        for layer in (e.layer2, e.layer3, e.layer4):
            f.append(layer(f[-1]))
        x = f[4]
        for i in range(4, -1, -1):
            x = torch.nn.functional.interpolate(self.up0[i](x), scale_factor=2, mode="nearest")
            if i > 0:
                x = torch.cat([x, f[i - 1]], 1)
            x = self.up1[i](x)
        return torch.sigmoid(self.disp(x))


def _resnet18_monodepth2(dev):
    """Deterministic fp32 cuDNN as for the stand-in network; seeded initialisation."""
    _tiny(dev)                                              # sets the cuDNN determinism flags
    torch.manual_seed(0)
    return _Monodepth2ResNet18().to(dev)


@pytest.mark.parametrize("net, dists", [("tiny", range(5, 10, 2)), ("resnet18", range(5, 10, 2)),
                                        ("tiny", range(5, 31, 2))], ids=["tiny", "resnet18", "tiny-far"])
def test_attack_classes_vs_oracle_loop_same_device(dev, calib, net, dists):
    """Our attack classes against the oracle's restatement of the reference loops, BOTH driven on the GPU with
    the same network, so the only difference is kernels vs torch ops.  `resnet18`: the random-init ResNet-18
    monodepth2 encoder / decoder BASELINE.json names (_Monodepth2ResNet18).  `tiny-far`: the classes' own default
    distances, 5-29 m."""
    import os
    from depthmodelhardening_b200 import attacks
    attacks.object_dataset_root = os.path.dirname(os.path.dirname(os.path.dirname(calib)))
    pbt = synth.patch_batch(batch=3, seed=4).to(dev)
    model = (_tiny(dev) if net == "tiny" else _resnet18_monodepth2(dev)).eval()
    # fraction of elements allowed to differ: sign(grad) flips where |grad| ~ 0.  The random-init ResNet-18 has far
    # more near-zero patch gradients than the 2-conv stand-in (measured 0.8 % over 3 L-inf steps against 0.1 %, with
    # the reference project's own ResnetEncoder / DepthDecoder, whose seeded weights differ from _Monodepth2ResNet18's)
    flips = 5e-3 if net == "tiny" else 2e-2
    l0_atol = 1e-4
    dist, ang = list(dists), list(range(-30, 31, 5))
    # ---- L-inf, 3 steps
    pl, fin = _placements(9, 3, (dist, ang), 3)
    ref = OQ.linf_attack(model, pbt.obj, pbt.mask, pbt.scenes, pl, fin, P34, eps=0.1, alpha=0.02)
    random.seed(9)
    atk = attacks.Phy_obj_atk(model, pbt.obj.clone(), pbt.mask.clone(), eps=0.1, alpha=0.02, steps=3,
                              random_start=False, dist_range=dist)
    out = atk(pbt.scenes.clone(), 3)
    assert float(((out[3] - ref[3]).abs() > 1e-6).float().mean()) < flips      # sign flips at |grad| ~ 0
    assert_close(out[1], ref[1], TOL, "benign scenes")
    assert_close(out[2], ref[2], TOL, "masks")
    if net == "resnet18":
        # L0 through this network is not a kernel test: |d cost / d patch| is ~1e-9 for most elements, below Adam's
        # eps = 1e-8, so the update lr * m / (sqrt(v) + eps) is LINEAR in grad / 1e-8 and iterating it amplifies the
        # 1e-5-level difference between the fused and the composed backward into O(0.1) pattern differences within 4
        # steps (measured with the reference project's network classes: 16 % of the elements beyond 5e-3) -- in both
        # directions, also between two torch runs with different cuDNN algorithms.  What IS checked with the real
        # network: one gradient of the attack cost w.r.t. the patch through fused apply -> ResNet-18 -> MSE against the
        # composed torch ops, same placements.
        from depthmodelhardening_b200 import patch_ops
        z0, al = pl[0]
        obj_a = pbt.obj.clone().requires_grad_(True)
        coeffs = patch_ops.homographies(z0, al, P34, obj_hw=(synth.PATCH_H, synth.PATCH_W)).to(dev)
        adv_a, m_a = patch_ops.apply_patch(obj_a, pbt.mask, pbt.scenes, coeffs)
        torch.nn.functional.mse_loss(model(adv_a) * m_a, torch.zeros_like(m_a)).backward()
        obj_b = pbt.obj.clone().requires_grad_(True)
        adv_b, m_b = OQ.apply_patch(obj_b, pbt.mask, pbt.scenes, z0, al, P34)
        torch.nn.functional.mse_loss(model(adv_b) * m_b, torch.zeros_like(m_b)).backward()
        assert_close(adv_a, adv_b, TOL, "adv scenes (ResNet-18 run)", max_outlier_frac=1e-4, outlier_rtol=1.0)
        assert_close(obj_a.grad, obj_b.grad, 5e-3, "d cost / d patch through ResNet-18")
        return
    # ---- L0, steps=2 (4 iterations)
    np.random.seed(3)
    init = [torch.Tensor(np.clip(np.random.random(pbt.obj.size()), 0.0, 1.0)).to(dev) for _ in range(2)]
    pl, fin = _placements(10, 4, (dist, ang), 3)
    ref0 = OQ.l0_attack(model, pbt.obj, pbt.mask, pbt.scenes, init[0], init[1], pl, fin, P34, steps=2, lr=0.5,
                        mask_wt=0.06, l0_thresh=0.1)
    random.seed(10)
    np.random.seed(3)
    atk0 = attacks.Phy_obj_atk_l0(model, pbt.obj.clone(), pbt.mask.clone(), adam_lr=0.5, steps=2, mask_wt=0.06,
                                  l0_thresh=0.1, dist_range=dist)
    out0 = atk0(pbt.scenes.clone(), 3)
    assert float(((atk0.pattern_pos_tensor - ref0[3]).abs() > l0_atol).float().mean()) < flips
    assert float(((atk0.pattern_neg_tensor - ref0[4]).abs() > l0_atol).float().mean()) < flips
    surv, surv_ref = (atk0.pattern.abs().sum(1) != 0), (ref0[5].abs().sum(1) != 0)
    assert float((surv != surv_ref).float().mean()) < flips


def test_batch_arena_roundtrip(dev):
    """staging.BatchArena: one pinned arena, one H2D copy; device views carry exactly the host values."""
    from depthmodelhardening_b200.staging import BatchArena
    ex = {("color", 0, 0): torch.rand(2, 3, 8, 12), ("K",): torch.rand(2, 4, 4), ("idx",): torch.arange(7, dtype=torch.int32),
          ("disp", 1): torch.rand(2, 1, 4, 6)}
    arena = BatchArena(ex, dev, slots=2)
    for k, v in arena.host_views(1).items():            # every slot has its own pinned buffer
        assert v.is_pinned() and v.shape == ex[k].shape and v.dtype == ex[k].dtype
        v.copy_(ex[k])
    arena.upload(1)
    assert arena.host_views(1)[("K",)].data_ptr() != arena.host_views(0)[("K",)].data_ptr()
    torch.cuda.synchronize()
    for k, v in arena.device_views(1).items():
        assert v.is_cuda and torch.equal(v.cpu(), ex[k])
        assert v.data_ptr() % 256 == 0


@pytest.mark.parametrize("n", [0, 1, 15, 16, 17, 256 * 3 + 5, 2 * 3 * 37 * 53])
def test_unpack_u8_is_to_tensor_bit_for_bit(dev, n):
    """8-bit frame transport (staging.unpack_u8 / dmh_unpack_u8): the device conversion equals torchvision's
    `to_tensor` arithmetic (`.to(float32).div(255)` on the CPU: IEEE division) bit for bit, for every byte value,
    ragged sizes (tail of n % 16 elements) and through a BatchArena slot."""
    from depthmodelhardening_b200.staging import BatchArena, unpack_u8
    g = torch.Generator().manual_seed(5 + n)
    src = torch.randint(0, 256, (n,), dtype=torch.uint8, generator=g)
    if n >= 256:
        src[:256] = torch.arange(256, dtype=torch.uint8)          # every value at least once
    ref = src.to(torch.float32).div(255)
    out = unpack_u8(src.to(dev))
    assert out.dtype == torch.float32 and torch.equal(out.cpu(), ref)
    if n == 2 * 3 * 37 * 53:
        ex = {("color", 0, 0): src.view(2, 3, 37, 53), ("K",): torch.rand(2, 4, 4)}
        arena = BatchArena(ex, dev, slots=1)
        for k, v in arena.host_views().items():
            v.copy_(ex[k])
        arena.upload(0)
        pre = torch.empty(2, 3, 37, 53, device=dev)
        got = unpack_u8(arena.device_views(0)[("color", 0, 0)], out=pre)
        assert got.data_ptr() == pre.data_ptr() and torch.equal(got.cpu(), ref.view(2, 3, 37, 53))
    with pytest.raises(RuntimeError):
        unpack_u8(torch.zeros(4, device=dev))                       # not uint8
    with pytest.raises(RuntimeError):
        unpack_u8(src)                                              # CPU tensor: no fallback


@pytest.mark.parametrize("ev", [False, True])
def test_vanila_attack_class_vs_reference_golden(dev, calib, ev):
    """Drop-in `Phy_obj_atk_vanila` (next-4: the placement-only attack of the evaluation harness) against the
    unmodified reference class run on the CPU (oracle/make_golden_vanila.py): same `random.sample` order -> same
    placements; adversarial / benign scenes and resized masks to fp32 tolerance."""
    import os
    from depthmodelhardening_b200 import attacks
    g = load_golden("attack_vanila")
    tag = "eval" if ev else "rand"
    attacks.object_dataset_root = os.path.dirname(os.path.dirname(os.path.dirname(calib)))
    pbt = synth.patch_batch(batch=3, seed=0).to(dev)
    other = synth.rand((1, 3, synth.PATCH_H, synth.PATCH_W), 77).to(dev)
    random.seed(11)
    atk = attacks.Phy_obj_atk_vanila(_tiny(dev), pbt.obj.clone(), pbt.mask.clone(), dist_range=list(range(5, 10, 2)))
    adv_s, ben_s, m_out, obj_adv = atk(pbt.scenes.clone(), other.clone(), 3, eval=ev)
    assert adv_s.shape == (3, 3, 320, 1024) and ben_s.shape == adv_s.shape and m_out.shape == (3, 1, 320, 1024)
    assert torch.equal(obj_adv, other)
    assert_close(m_out.double().sum(), g[tag + "_mask_sum"], 1e-6)
    assert_close(adv_s.double().sum(), g[tag + "_adv_sum"], 1e-6)
    assert_close(ben_s.double().sum(), g[tag + "_ben_sum"], 1e-6)
    assert_close(adv_s[:, :, 90:200:2, 380:640:2], g[tag + "_adv_crop"], TOL, "adv crop")
    assert_close(ben_s[:, :, 90:200:2, 380:640:2], g[tag + "_ben_crop"], TOL, "ben crop")
    assert_close(m_out[:, :, 90:200:2, 380:640:2], g[tag + "_mask_crop"], TOL, "mask crop")
    with pytest.raises(RuntimeError, match="Batch size"):
        atk(pbt.scenes[:2].clone(), other.clone(), 3)
