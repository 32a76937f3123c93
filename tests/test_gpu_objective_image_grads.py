"""GPU: gradients of the fused objective (ops.objective, objective.photometric_losses) w.r.t. the colour frames --
the target colour(0, 0), the pyramid colour(0, s) and every source frame -- against the autograd gradients of the
fp32 oracle, arbitrated by its fp64 run.  Every case also checks that asking for them leaves the losses, the
disparity gradients and the pose gradients bit for bit as they are without them."""
import types

import pytest
import torch

from depthmodelhardening_b200 import objective, synth
from oracle import photometric as OP
from tests.util import assert_close, assert_grad_close

pytestmark = pytest.mark.gpu
TOL = 1e-5
OUTL = 2e-3
# A pixel whose automask / argmin decision falls the other way than in the oracle (a float near-tie, see
# assert_selection_close) moves the gradient of every element its 3x3 window touches: 9 pixels x 3 channels, each
# scattered to up to 4 bilinear taps in a source frame.
FLIP_FOOTPRINT = 9 * 3 * 4


@pytest.fixture(scope="module")
def dev():
    from depthmodelhardening_b200 import _lib
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    _lib.load()
    return torch.device("cuda:0")


def _colour_keys(pb):
    return [(0, s) for s in pb.scales] + [(f, 0) for f in pb.frame_ids[1:]]


def _oracle(pb, over, dtype, keys, up=None):
    colors = {k: v.detach().to(dtype) for k, v in pb.color.items()}
    for k in keys:
        colors[k].requires_grad_(True)
    disps = {s: v.detach().to(dtype) for s, v in pb.disp.items()}
    opts = OP.default_opts(scales=list(pb.scales), min_depth=pb.min_depth, max_depth=pb.max_depth, **over)
    total, losses, aux = OP.photometric_objective(colors, disps, pb.K.to(dtype), pb.inv_K.to(dtype),
                                                  {k: v.to(dtype) for k, v in pb.T.items()}, pb.frame_ids,
                                                  {k: v.to(dtype) for k, v in pb.noise.items()}, opts, return_aux=True)
    _weighted(total, losses, pb.scales, up).backward()
    grads = {k: colors[k].grad for k in keys}
    grads["argmin"] = {s: aux[("argmin", s)] for s in pb.scales if ("argmin", s) in aux}
    return grads


def _weighted(total, losses, scales, up):
    if up is None:
        return total
    out = total * up[0]
    for i, s in enumerate(scales):
        out = out + losses["loss/%d" % s] * up[1 + i]
    return out


def _fused(pb, dev, over, keys, want_T=False, up=None, dtype=None, sel=None):
    g = pb.to(dev)
    colors = {k: (v.to(dtype) if dtype is not None else v).clone() for k, v in g.color.items()}
    for k in keys:
        colors[k].requires_grad_(True)
    disps = {s: g.disp[s].clone().requires_grad_(True) for s in g.scales}
    Ts = {k: v.clone().requires_grad_(want_T and k != "s") for k, v in g.T.items()}
    losses, aux = objective.photometric_losses(
        colors, disps, g.K, g.inv_K, Ts, g.frame_ids, g.scales, g.height, g.width,
        no_ssim=bool(over.get("no_ssim")), avg_reprojection=bool(over.get("avg_reprojection")),
        disable_automasking=bool(over.get("disable_automasking")), noise=g.noise, want_selection=sel is not None)
    if sel is not None:
        sel.update({s: aux[("argmin", s)].cpu() for s in g.scales})
    _weighted(losses["loss"], {k: v for k, v in losses.items()}, g.scales, up).backward()
    return (losses, {s: d.grad for s, d in disps.items()}, {k: t.grad for k, t in Ts.items() if t.requires_grad},
            {k: colors[k].grad for k in colors})


def _flips(sel, ref):
    """pixels whose decision differs from the oracle's, over all scales"""
    return sum(int((sel[s] != ref[s].to(sel[s].dtype)).sum()) for s in ref)


def _assert_colour_grad(g, ref32, ref64, rtol, what, flips):
    assert_grad_close(g, ref32, ref64, rtol, what, outlier_frac=OUTL + flips * FLIP_FOOTPRINT / g.numel())


def _check(pb, dev, over, keys=None, want_T=False, up=None):
    keys = _colour_keys(pb) if keys is None else keys
    sel = {}
    losses, gd, gT, gc = _fused(pb, dev, over, keys, want_T, up, sel=sel)
    losses0, gd0, gT0, gc0 = _fused(pb, dev, over, [], want_T, up)
    for k in losses0:
        assert torch.equal(losses[k], losses0[k]), k
    for s in gd0:
        assert torch.equal(gd[s], gd0[s]), "grad_disp %d" % s
    for f in gT0:
        assert torch.equal(gT[f], gT0[f]), "grad_T %s" % f
    ref32 = _oracle(pb, over, torch.float32, keys, up)
    ref64 = _oracle(pb, over, torch.float64, keys, up)
    flips = _flips(sel, ref32["argmin"])
    for k in pb.color:
        if k in keys:
            assert gc[k] is not None and gc[k].dtype == torch.float32, k
            _assert_colour_grad(gc[k], ref32[k], ref64[k], TOL, "grad colour %s" % (k,), flips)
        else:
            assert gc[k] is None, k
    return gc


@pytest.mark.parametrize("frame_ids,shape,want_T", [((0, "s"), (4, 192, 640), False),
                                                    ((0, "s"), (2, 320, 1024), False),
                                                    ((0, -1, 1), (2, 96, 320), True),
                                                    ((0, -1, 1, "s"), (1, 72, 200), True),
                                                    ((0, "s"), (2, 50, 70), False)])
def test_colour_grads_vs_oracle(dev, frame_ids, shape, want_T):
    """Config 1 (B=4, 640x192), the benchmarked instantiation (1024x320, all scales in one launch), three and four
    frames with pose gradients (the multi-source kernel), and a ragged size with W % 4 != 0 (general kernel)."""
    B, H, W = shape
    scales = (0, 1, 2, 3) if H % 8 == 0 and W % 8 == 0 else (0, 1)
    pb = synth.photo_batch(batch=B, height=H, width=W, frame_ids=frame_ids, scales=scales, seed=41)
    _check(pb, dev, {}, want_T=want_T)


@pytest.mark.parametrize("frame_ids,over", [((0, "s"), dict(disable_automasking=True)),
                                            ((0, -1, 1), dict(disable_automasking=True)),
                                            ((0, -1, 1), dict(avg_reprojection=True)),
                                            ((0, -1, 1), dict(avg_reprojection=True, disable_automasking=True)),
                                            ((0, "s"), dict(no_ssim=True))])
def test_colour_grads_options(dev, frame_ids, over):
    pb = synth.photo_batch(batch=2, height=64, width=96, frame_ids=frame_ids, seed=43)
    _check(pb, dev, over)


def test_colour_grads_per_scale_upstream(dev):
    """Distinct upstream weights on `loss` and on every `loss/s`."""
    pb = synth.photo_batch(batch=2, height=64, width=96, frame_ids=(0, -1, 1), seed=45)
    _check(pb, dev, {}, up=[0.7, 1.3, -0.4, 2.0, 0.25])


@pytest.mark.parametrize("which", ["target", "source", "pyramid"])
def test_colour_grads_subsets(dev, which):
    """Only one colour input requires grad: it matches the oracle, every other keeps .grad None."""
    pb = synth.photo_batch(batch=2, height=64, width=96, frame_ids=(0, -1, 1), seed=47)
    keys = {"target": [(0, 0)], "source": [(1, 0)], "pyramid": [(0, 2)]}[which]
    _check(pb, dev, {}, keys=keys)


def test_colour_grads_full_size_properties(dev):
    """B=8 of 1024x320: the target and pyramid gradients are bit-identical over two runs (the source gradients are
    scattered atomically: equal to 1e-6 of their maximum); a 3x upstream gives 3x the gradients (to 1e-5 of their
    maximum: the terms of the SSIM coefficient form cancel, so each rounding counts relative to the larger terms)."""
    pb = synth.photo_batch(batch=8, height=320, width=1024, frame_ids=(0, "s"), seed=49)
    keys = _colour_keys(pb)
    _, _, _, a = _fused(pb, dev, {}, keys)
    _, _, _, b = _fused(pb, dev, {}, keys)
    _, _, _, c = _fused(pb, dev, {}, keys, up=[3.0] + [0.0] * len(pb.scales))
    for k in keys:
        if k[0] == 0:
            assert torch.equal(a[k], b[k]), k
        else:
            assert_close(b[k], a[k], 1e-6, "source %s rerun" % (k,))
        assert float(a[k].abs().max()) > 0, k
        assert_close(c[k], 3.0 * a[k], TOL, "3x upstream %s" % (k,))


def test_colour_grads_cuda_graph_replay(dev):
    """Forward + backward (colour and disparity gradients) captured in a CUDA graph and replayed equals eager."""
    pb = synth.photo_batch(batch=2, height=64, width=96, frame_ids=(0, -1, 1), seed=51)
    g = pb.to(dev)
    keys = _colour_keys(pb)
    colors = {k: v.clone().requires_grad_(k in keys) for k, v in g.color.items()}
    disps = {s: v.clone().requires_grad_(True) for s, v in g.disp.items()}
    ins = [colors[k] for k in keys] + [disps[s] for s in g.scales]

    def run():
        losses, _ = objective.photometric_losses(colors, disps, g.K, g.inv_K, g.T, g.frame_ids, g.scales, g.height,
                                                 g.width, noise=g.noise)
        return torch.autograd.grad(losses["loss"], ins)

    eager = [t.clone() for t in run()]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        run()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static = run()
    graph.replay()
    torch.cuda.synchronize()
    for i, (e, r) in enumerate(zip(eager, static)):
        assert_close(r, e, 1e-6, "graph replay input %d" % i)


def test_colour_grads_bf16_frames(dev):
    """bf16 frames: gradients come back in bf16, within the bf16 class of the oracle on the rounded frames."""
    pb = synth.photo_batch(batch=2, height=64, width=96, frame_ids=(0, "s"), seed=53)
    for k in list(pb.color):
        pb.color[k] = pb.color[k].to(torch.bfloat16).float()
    keys = _colour_keys(pb)
    sel = {}
    _, _, _, gc = _fused(pb, dev, {}, keys, dtype=torch.bfloat16, sel=sel)
    ref32 = _oracle(pb, {}, torch.float32, keys)
    ref64 = _oracle(pb, {}, torch.float64, keys)
    flips = _flips(sel, ref32["argmin"])
    for k in keys:
        assert gc[k].dtype == torch.bfloat16, k
        _assert_colour_grad(gc[k].float(), ref32[k], ref64[k], 4e-3, "bf16 grad colour %s" % (k,), flips)


def test_fused_compute_losses_colour_grads(dev):
    """The patched Trainer.compute_losses on a namespace trainer: inputs[("color", f, s)] requiring grad receive the
    oracle's gradients."""
    pb = synth.photo_batch(batch=2, height=64, width=96, frame_ids=(0, -1, "s"), seed=55)
    g = pb.to(dev)
    opt = types.SimpleNamespace(v1_multiscale=False, pose_model_type="separate_resnet", predictive_mask=False,
                                adv_train=False, scales=list(g.scales), frame_ids=list(g.frame_ids), height=g.height,
                                width=g.width, min_depth=pb.min_depth, max_depth=pb.max_depth, no_ssim=False,
                                avg_reprojection=False, disable_automasking=False, disparity_smoothness=1e-3)
    trainer = types.SimpleNamespace(opt=opt, _dmh_noise=g.noise)
    inputs = {("color", f, s): v.clone().requires_grad_(True) for (f, s), v in g.color.items()}
    inputs[("K", 0)], inputs[("inv_K", 0)], inputs["stereo_T"] = g.K, g.inv_K, g.T["s"]
    outputs = {("disp", s): g.disp[s].clone().requires_grad_(True) for s in g.scales}
    outputs[("cam_T_cam", 0, -1)] = g.T[-1]
    losses = objective.fused_compute_losses(trainer, inputs, outputs)
    losses["loss"].backward()
    keys = _colour_keys(pb)
    ref32 = _oracle(pb, {}, torch.float32, keys)
    ref64 = _oracle(pb, {}, torch.float64, keys)
    for (f, s) in keys:
        assert_grad_close(inputs[("color", f, s)].grad, ref32[(f, s)], ref64[(f, s)], TOL, "color %s %s" % (f, s),
                          outlier_frac=OUTL)
