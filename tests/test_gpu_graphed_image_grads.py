"""Frame and pose gradients of the two entry points that gained them last:

- objective.GraphedObjective, the CUDA-graph replay of forward + backward, for the monodepth2 objective and for the
  depth-hints objective: every gradient it returns equals the eager path's on the same inputs, over three replays with
  new inputs copied in between.
- ops.photo_scale_sum (one scale, full resolution): d(sum)/d(target), d(sum)/d(source f) and d(sum)/d(ident) against
  the autograd gradients of the fp32 oracle, arbitrated by its fp64 run.

The source-frame gradients are scattered through the bilinear taps with atomic adds, so their last bits depend on the
order the adds land in: they are compared to 1e-6 of their maximum.  Everything else is compared bit for bit."""
import pytest
import torch
import torch.nn.functional as F

from depthmodelhardening_b200 import depth_hints as DH
from depthmodelhardening_b200 import objective, ops, synth
from oracle import photometric as OP
from tests.util import assert_close, assert_grad_close

gpu = pytest.mark.gpu
TOL = 1e-5
OUTL = 2e-3
# a pixel whose argmin falls the other way than in the oracle moves the gradient of every element its 3x3 window
# touches: 9 pixels x 3 channels, each scattered to up to 4 bilinear taps in a source frame
FLIP_FOOTPRINT = 9 * 3 * 4


@pytest.fixture(scope="module")
def dev():
    from depthmodelhardening_b200 import _lib
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    _lib.load()
    return torch.device("cuda:0")


def _assert_grad_equal(a, b, what, source):
    assert a.dtype == b.dtype, what
    if source:
        assert_close(a, b, 1e-6, what)
    else:
        assert torch.equal(a, b), what


# ----------------------------------------------------------------------------------------------- GraphedObjective
def _batch(frame_ids, seed, hints):
    return synth.photo_batch(batch=4, height=96, width=160, frame_ids=frame_ids, seed=seed, depth_hints=hints)


def _eager(pb, cols, poses, hints, over, dtype=None):
    colors = {k: (v.to(dtype) if dtype is not None else v).clone().requires_grad_(k in cols)
              for k, v in pb.color.items()}
    disps = {s: pb.disp[s].clone().requires_grad_(True) for s in pb.scales}
    Ts = {f: t.clone().requires_grad_(f in poses) for f, t in pb.T.items()}
    if hints is None:
        losses, _ = objective.photometric_losses(colors, disps, pb.K, pb.inv_K, Ts, pb.frame_ids, pb.scales, pb.height,
                                                 pb.width, noise=pb.noise, **over)
    else:
        noise = {s: pb.noise[s][:, :1].contiguous() for s in pb.scales}
        losses, _ = DH.depth_hint_losses(colors, disps, pb.K, pb.inv_K, Ts, pb.frame_ids, pb.scales, pb.height,
                                         pb.width, pb.extras["depth_hint"], pb.extras["depth_hint_mask"], hints,
                                         noise=noise, fused=True, **over)
    losses["loss"].backward()
    grads = {s: disps[s].grad for s in pb.scales}
    grads.update({("color",) + k: colors[k].grad for k in cols})
    grads.update({("T", f): Ts[f].grad for f in poses})
    return {k: v.detach().clone() for k, v in losses.items()}, grads


def _graphed_vs_eager(dev, frame_ids, cols, poses, hints=None, over=None, dtype=None):
    over = dict(over or {})
    dh = hints is not None
    a, b = (_batch(frame_ids, seed, dh).to(dev) for seed in (61, 62))
    colors = {k: (v.to(dtype) if dtype is not None else v).clone().requires_grad_(k in cols) for k, v in a.color.items()}
    Ts = {f: t.clone().requires_grad_(f in poses) for f, t in a.T.items()}
    extra = dict(depth_hint=a.extras["depth_hint"], depth_hint_mask=a.extras["depth_hint_mask"],
                 use_depth_hints=hints) if dh else {}
    g = objective.GraphedObjective(colors, a.disp, a.K, a.inv_K, Ts, a.frame_ids, a.scales, a.height, a.width,
                                   noise=a.noise, **extra, **over)
    expect = set(a.scales) | {("color",) + k for k in cols} | {("T", f) for f in poses}
    for pb in (a, b, a):
        kw = dict(depth_hint=pb.extras["depth_hint"], depth_hint_mask=pb.extras["depth_hint_mask"]) if dh else {}
        colors = {k: (v.to(dtype) if dtype is not None else v) for k, v in pb.color.items()}
        losses, grads = g(colors, pb.disp, pb.K, pb.inv_K, pb.T, pb.noise, **kw)
        torch.cuda.synchronize()
        l_ref, g_ref = _eager(pb, cols, poses, hints, over, dtype)
        for k in l_ref:
            assert torch.equal(losses[k], l_ref[k]), k
        assert set(grads) == expect
        for k in expect:
            assert g_ref[k] is not None and float(g_ref[k].abs().max()) > 0, k
            frame = isinstance(k, tuple) and k[0] == "color"
            _assert_grad_equal(grads[k], g_ref[k], "grad %s" % (k,), frame and k[1] != 0)
            if frame and dtype is not None:
                assert grads[k].dtype == dtype, k


ALL2 = [(0, 0), (0, 1), (0, 2), (0, 3), ("s", 0)]
ALL3 = [(0, 0), (0, 1), (0, 2), (0, 3), (-1, 0), (1, 0)]
ALL4 = ALL3 + [("s", 0)]


@gpu
@pytest.mark.parametrize("frame_ids,cols,poses", [
    ((0, "s"), ALL2, []),
    ((0, "s"), [], ["s"]),
    ((0, "s"), [(0, 0), ("s", 0)], ["s"]),
    ((0, -1, 1), ALL3, [-1, 1]),
    ((0, -1, 1), [(0, 2), (1, 0)], []),
    ((0, -1, 1, "s"), ALL4, [-1, 1]),
    ((0, -1, 1, "s"), [], [-1, 1]),
    ((0, -1, 1, "s"), [(0, 0), (-1, 0)], [1]),
], ids=["s-frames", "s-pose", "s-both", "m-both", "m-subset", "ms-both", "ms-poses", "ms-subset"])
def test_graphed_objective_grads_match_eager(dev, frame_ids, cols, poses):
    """monodepth2 objective: stereo, mono and mono+stereo, with frames, poses, both or a subset marked."""
    _graphed_vs_eager(dev, frame_ids, cols, poses)


@gpu
def test_graphed_objective_grads_options(dev):
    """avg_reprojection and no_ssim take the general per-scale kernel; one identity plane under avg_reprojection."""
    _graphed_vs_eager(dev, (0, -1, 1), ALL3, [-1], over=dict(avg_reprojection=True))
    _graphed_vs_eager(dev, (0, "s"), ALL2, [], over=dict(no_ssim=True))


@gpu
def test_graphed_objective_nothing_marked(dev):
    """With no frame or pose marked, the replay returns the disparity gradients only, as eager."""
    _graphed_vs_eager(dev, (0, -1, 1, "s"), [], [])


@gpu
def test_graphed_objective_bf16_frames(dev):
    """bf16 frames: the frame gradients come back in bf16, equal to the eager bf16 path."""
    _graphed_vs_eager(dev, (0, "s"), ALL2, [], dtype=torch.bfloat16)


@gpu
@pytest.mark.parametrize("hints", [True, False], ids=["hints", "no-hints"])
@pytest.mark.parametrize("frame_ids,cols,poses", [((0, "s"), ALL2, []), ((0, -1, 1, "s"), ALL4, [-1, 1])],
                         ids=["s", "ms"])
def test_graphed_depth_hints_grads_match_eager(dev, frame_ids, cols, poses, hints):
    """depth-hints objective: stereo only (the single-source fast kernel) and mono+stereo (the general kernel, pose
    gradients), with and without use_depth_hints."""
    _graphed_vs_eager(dev, frame_ids, cols, poses, hints=hints)


def test_graphed_objective_rejects_foreign_options():
    """An option only the other objective accepts is refused before anything runs."""
    t = torch.zeros(1)
    with pytest.raises(TypeError, match="use_depth_hints"):
        objective.GraphedObjective({(0, 0): t}, {}, t, t, {}, [0, "s"], [0], 8, 8, use_depth_hints=True)
    with pytest.raises(TypeError, match="fused"):
        objective.GraphedObjective({(0, 0): t}, {}, t, t, {}, [0, "s"], [0], 8, 8, depth_hint=t, depth_hint_mask=t,
                                   fused=False)
    with pytest.raises(ValueError, match="together"):
        objective.GraphedObjective({(0, 0): t}, {}, t, t, {}, [0, "s"], [0], 8, 8, depth_hint=t)


# ------------------------------------------------------------------------------------------------ photo_scale_sum
def _sum_case(frame_ids, hw, over, seed=71, down=False):
    H, W = hw
    pb = synth.photo_batch(batch=2, height=H, width=W, frame_ids=frame_ids, scales=(0, 1), seed=seed)
    srcs_ids = pb.frame_ids[1:]
    disp = F.interpolate(pb.disp[1], (H, W), mode="bilinear", align_corners=False) if down else pb.disp[0]
    if over.get("input_is_depth"):
        disp = OP.disp_to_depth(disp, 0.1, 100.0)[1]
    ident = None
    if not over.get("no_ident"):
        ident = torch.cat([OP.reprojection_loss(pb.color[(f, 0)], pb.color[(0, 0)], bool(over.get("no_ssim")))
                           for f in srcs_ids], 1).detach()
    noise = pb.noise[0][:, :1].contiguous() if over.get("avg_reprojection") else pb.noise[0]
    return pb, srcs_ids, disp.contiguous(), ident, noise


def _sum_oracle(pb, srcs_ids, disp, ident, noise, over, dtype, up=1.0):
    dt = lambda t: t.detach().to(dtype)
    tg = dt(pb.color[(0, 0)]).requires_grad_(True)
    srcs = [dt(pb.color[(f, 0)]).requires_grad_(True) for f in srcs_ids]
    K, inv_K, d = dt(pb.K), dt(pb.inv_K), dt(disp)
    rp = []
    for f, src in zip(srcs_ids, srcs):
        if over.get("input_is_depth"):
            grid = OP.project3d(OP.backproject(d, inv_K), K, dt(pb.T[f]), pb.height, pb.width)
            pred = OP.warp(src, grid)
        else:
            pred = OP.warp_from_disp(d, src, K, inv_K, dt(pb.T[f]), 0.1, 100.0)[0]
        rp.append(OP.reprojection_loss(pred, tg, bool(over.get("no_ssim"))))
    reproj = torch.cat(rp, 1)
    idn = dt(ident).requires_grad_(True) if ident is not None else None
    if over.get("avg_reprojection"):
        reproj = reproj.mean(1, True)
    comb = reproj
    if idn is not None:
        iv = idn.mean(1, True) if over.get("avg_reprojection") else idn
        comb = torch.cat((iv + dt(noise), reproj), 1)
    to_opt, idx = torch.min(comb, dim=1)
    (to_opt.sum() * up).backward()
    out = {"target": tg.grad, "argmin": idx}
    out.update({f: s.grad for f, s in zip(srcs_ids, srcs)})
    if idn is not None:
        out["ident"] = idn.grad
    return out


def _sum_cuda(pb, srcs_ids, disp, ident, noise, over, dev, marked=True, dtype=None, up=1.0, want_T=False):
    g = pb.to(dev)
    cast = lambda t: (t.to(dtype) if dtype is not None else t).clone().requires_grad_(marked)
    tg = cast(g.color[(0, 0)])
    srcs = [cast(g.color[(f, 0)]) for f in srcs_ids]
    idn = ident.to(dev).requires_grad_(marked) if ident is not None else None
    d = disp.to(dev).requires_grad_(True)
    Ts = [g.T[f].clone().requires_grad_(want_T) for f in srcs_ids]
    total, sel = ops.photo_scale_sum(d, tg, srcs, Ts, g.K, g.inv_K, ident=idn,
                                     noise=noise.to(dev) if ident is not None else None,
                                     no_ssim=bool(over.get("no_ssim")), avg_reprojection=bool(over.get("avg_reprojection")),
                                     input_is_depth=bool(over.get("input_is_depth")), want_sel=True)
    (total * up).backward()
    out = {"total": total.detach(), "sel": sel, "disp": d.grad, "target": tg.grad}
    out.update({f: s.grad for f, s in zip(srcs_ids, srcs)})
    out.update({("T", f): t.grad for f, t in zip(srcs_ids, Ts) if want_T})
    if idn is not None:
        out["ident"] = idn.grad
    return out


SUM_CASES = {
    "stereo": ((0, "s"), (64, 96), {}, False),
    "no_ssim": ((0, "s"), (64, 96), {"no_ssim": True}, False),
    "three-sources": ((0, -1, 1, "s"), (64, 96), {}, False),
    "avg": ((0, -1, 1), (64, 96), {"avg_reprojection": True}, False),
    "avg-one-source": ((0, "s"), (64, 96), {"avg_reprojection": True}, False),
    "depth": ((0, "s"), (64, 96), {"input_is_depth": True}, False),
    "depth-three-sources": ((0, -1, 1, "s"), (64, 96), {"input_is_depth": True}, False),
    "no-ident": ((0, -1, 1), (64, 96), {"no_ident": True}, False),
    "ragged": ((0, -1, 1), (33, 37), {}, False),
    "down-sampled-disp": ((0, -1, 1), (64, 96), {}, True),
}


@gpu
@pytest.mark.parametrize("name", sorted(SUM_CASES))
def test_photo_scale_sum_grads_vs_oracle(dev, name):
    """Target, source and identity gradients against the oracle; asking for them leaves the sum, the selection, the
    disparity gradient and the pose gradients bit for bit as they are without them."""
    frame_ids, hw, over, down = SUM_CASES[name]
    pb, srcs_ids, disp, ident, noise = _sum_case(frame_ids, hw, over, down=down)
    want_T = frame_ids[1] != "s"
    got = _sum_cuda(pb, srcs_ids, disp, ident, noise, over, dev, want_T=want_T)
    base = _sum_cuda(pb, srcs_ids, disp, ident, noise, over, dev, marked=False, want_T=want_T)
    for k in ("total", "sel", "disp") + tuple(("T", f) for f in srcs_ids if want_T):
        assert torch.equal(got[k], base[k]), k
    ref32 = _sum_oracle(pb, srcs_ids, disp, ident, noise, over, torch.float32)
    ref64 = _sum_oracle(pb, srcs_ids, disp, ident, noise, over, torch.float64)
    flips = int((got["sel"].cpu() != ref32["argmin"].to(torch.uint8)).sum())
    keys = ["target"] + list(srcs_ids) + (["ident"] if ident is not None else [])
    for k in keys:
        assert got[k] is not None and got[k].dtype == torch.float32, k
        assert float(got[k].abs().max()) > 0, k
        assert_grad_close(got[k], ref32[k], ref64[k], TOL, "grad %s" % (k,),
                          outlier_frac=OUTL + flips * FLIP_FOOTPRINT / got[k].numel())


@gpu
def test_photo_scale_sum_bf16_frames(dev):
    """bf16 frames: the gradients come back in bf16, within the bf16 class of the oracle on the rounded frames."""
    pb, srcs_ids, disp, ident, noise = _sum_case((0, -1, 1), (64, 96), {}, seed=72)
    for k in list(pb.color):
        pb.color[k] = pb.color[k].to(torch.bfloat16).float()
    got = _sum_cuda(pb, srcs_ids, disp, ident, noise, {}, dev, dtype=torch.bfloat16)
    ref32 = _sum_oracle(pb, srcs_ids, disp, ident, noise, {}, torch.float32)
    ref64 = _sum_oracle(pb, srcs_ids, disp, ident, noise, {}, torch.float64)
    for k in ["target"] + list(srcs_ids):
        assert got[k].dtype == torch.bfloat16, k
        assert_grad_close(got[k].float(), ref32[k], ref64[k], 4e-3, "bf16 grad %s" % (k,), outlier_frac=OUTL)
    assert got["ident"].dtype == torch.float32


@gpu
def test_photo_scale_sum_grads_deterministic_and_linear(dev):
    """Two runs give the same target and identity gradients bit for bit (the sources to 1e-6); a 3x upstream
    gives 3x every gradient."""
    pb, srcs_ids, disp, ident, noise = _sum_case((0, -1, 1, "s"), (96, 160), {}, seed=73)
    a = _sum_cuda(pb, srcs_ids, disp, ident, noise, {}, dev)
    b = _sum_cuda(pb, srcs_ids, disp, ident, noise, {}, dev)
    c = _sum_cuda(pb, srcs_ids, disp, ident, noise, {}, dev, up=3.0)
    for k in ["target", "ident"] + list(srcs_ids):
        _assert_grad_equal(b[k], a[k], "rerun %s" % (k,), k not in ("target", "ident"))
        assert_close(c[k], 3.0 * a[k], TOL, "3x upstream %s" % (k,))
