"""GPU: gradients of the depth-hints objective (depth_hints.depth_hint_losses, both implementations) w.r.t. the colour
frames -- the target colour(0, 0), the pyramid colour(0, s) and every source frame -- against the autograd gradients
of the fp32 oracle (oracle/depth_hints.py), arbitrated by its fp64 run.  Every fused case also checks that asking for
them leaves the losses, the selections, the disparity gradients and the pose gradients bit for bit as they are
without them.  The last test checks the winning-source bits that dmh_photo_scale_dh records under
DMH_PHOTO_SEL_SOURCE, which route the reprojection gradient between several source frames."""
import types

import pytest
import torch
import torch.nn.functional as F

from depthmodelhardening_b200 import _lib, depth_hints as DH, ops, synth
from depthmodelhardening_b200._lib import check, ptr, ptr_array, stream
from oracle import depth_hints as OD
from oracle import photometric as OP
from oracle.make_golden_dh import CASES
from tests.util import assert_close, assert_grad_close

pytestmark = pytest.mark.gpu
TOL = 1e-5
OUTL = 2e-3
# A pixel whose argmin falls the other way than in the oracle (a float near-tie) moves the gradient of every element
# its 3x3 window touches: 9 pixels x 3 channels, each scattered to up to 4 bilinear taps in a source frame.
FLIP_FOOTPRINT = 9 * 3 * 4


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    _lib.load()
    return torch.device("cuda:0")


def _colour_keys(pb):
    return [(0, s) for s in pb.scales] + [(f, 0) for f in pb.frame_ids[1:]]


def _weighted(losses, scales, up, hints):
    """losses["loss"] * up[0] + sum_s of up[...] times loss/s, reproj_loss/s and (with hints) depth_hint_loss/s"""
    if up is None:
        return losses["loss"]
    out = losses["loss"] * up[0]
    i = 1
    for key in ("loss/%d", "reproj_loss/%d") + (("depth_hint_loss/%d",) if hints else ()):
        for s in scales:
            out = out + losses[key % s] * up[i]
            i += 1
    return out


def _oracle(pb, hints, over, dtype, keys, up=None):
    colors = {k: v.detach().to(dtype) for k, v in pb.color.items()}
    for k in keys:
        colors[k].requires_grad_(True)
    disps = {s: v.detach().to(dtype) for s, v in pb.disp.items()}
    opts = OP.default_opts(scales=list(pb.scales), min_depth=pb.min_depth, max_depth=pb.max_depth, **over)
    _, losses, aux = OD.depth_hints_objective(colors, disps, pb.K.to(dtype), pb.inv_K.to(dtype),
                                              {k: v.to(dtype) for k, v in pb.T.items()}, pb.frame_ids,
                                              {k: v[:, :1].to(dtype) for k, v in pb.noise.items()},
                                              pb.extras["depth_hint"].to(dtype), pb.extras["depth_hint_mask"].to(dtype),
                                              hints, opts, return_aux=True)
    _weighted(losses, pb.scales, up, hints).backward()
    grads = {k: colors[k].grad for k in keys}
    grads["argmin"] = {s: aux[("argmin", s)][:, 0] for s in pb.scales}
    return grads


def _run(pb, dev, hints, over, keys, want_T=False, up=None, fused=True, want_sel=True, dtype=None):
    g = pb.to(dev)
    colors = {k: (v.to(dtype) if dtype is not None else v).clone() for k, v in g.color.items()}
    for k in keys:
        colors[k].requires_grad_(True)
    disps = {s: g.disp[s].clone().requires_grad_(True) for s in g.scales}
    Ts = {k: v.clone().requires_grad_(want_T and k != "s") for k, v in g.T.items()}
    noise = {s: g.noise[s][:, :1].contiguous() for s in g.scales}
    losses, aux = DH.depth_hint_losses(colors, disps, g.K, g.inv_K, Ts, g.frame_ids, g.scales, g.height, g.width,
                                       g.extras["depth_hint"], g.extras["depth_hint_mask"], hints, g.min_depth,
                                       g.max_depth, noise=noise, want_selection=want_sel, fused=fused, **over)
    _weighted(losses, g.scales, up, hints).backward()
    return (losses, aux, {s: d.grad for s, d in disps.items()},
            {k: t.grad for k, t in Ts.items() if t.requires_grad}, {k: colors[k].grad for k in colors})


def _check(pb, dev, hints, over, keys=None, want_T=False, up=None, fused=True):
    keys = _colour_keys(pb) if keys is None else keys
    losses, aux, gd, gT, gc = _run(pb, dev, hints, over, keys, want_T, up, fused)
    if fused:
        losses0, aux0, gd0, gT0, _ = _run(pb, dev, hints, over, [], want_T, up, fused)
        for k in losses0:
            assert torch.equal(losses[k], losses0[k]), k
        for k in aux0:
            assert torch.equal(aux[k], aux0[k]), k
        for s in gd0:
            assert torch.equal(gd[s], gd0[s]), "grad_disp %d" % s
        for f in gT0:
            assert torch.equal(gT[f], gT0[f]), "grad_T %s" % f
    ref32 = _oracle(pb, hints, over, torch.float32, keys, up)
    ref64 = _oracle(pb, hints, over, torch.float64, keys, up)
    # the masked mean divides by sum(m_r): a flipped argmin rescales the scale's whole reprojection term
    # (test_depth_hints.test_cuda_matches_oracle_and_golden), and moves its own 3x3 footprint
    rtol, flips = TOL, 0
    for s in pb.scales:
        sel, ref = aux[("argmin", s)].cpu(), ref32["argmin"][s]
        assert int(sel.max()) <= 2, "argmin output carries the source bits"
        n = int((sel != ref.to(sel.dtype)).sum())
        flips += n
        rtol += n * 8.0 / max(int((ref != 1).sum()), 1)
    for k in pb.color:
        if k in keys:
            assert gc[k] is not None and gc[k].dtype == torch.float32, k
            assert float(gc[k].abs().max()) > 0, k
            assert_grad_close(gc[k], ref32[k], ref64[k], rtol, "grad colour %s" % (k,),
                              outlier_frac=OUTL + flips * FLIP_FOOTPRINT / gc[k].numel())
        else:
            assert gc[k] is None, k
    return gc


@pytest.mark.parametrize("fused", [True, False], ids=["fused", "oplevel"])
@pytest.mark.parametrize("name", sorted(CASES))
def test_colour_grads_vs_oracle(dev, name, fused):
    """The five golden configurations (stereo F=1 on the fast kernel, mono+stereo F=3 on the general kernel with the
    winning-source bits, no hints, avg_reprojection, no_ssim), through both implementations."""
    skw, hints, over = CASES[name]
    _check(synth.photo_batch(**skw), dev, hints, over, fused=fused)


@pytest.mark.parametrize("frame_ids", [(0, "s"), (0, -1, 1)])
def test_colour_grads_no_automask(dev, frame_ids):
    """disable_automasking (only without hints: the reference raises with both): every pixel's reprojection counts."""
    pb = synth.photo_batch(batch=2, height=64, width=96, frame_ids=frame_ids, seed=61, depth_hints=True)
    _check(pb, dev, False, dict(disable_automasking=True))


@pytest.mark.parametrize("frame_ids", [(0, "s"), (0, -1, 1, "s")])
def test_colour_grads_with_pose_grads(dev, frame_ids):
    """Pose gradients on T (the general kernel, also for one source) together with the colour gradients."""
    pb = synth.photo_batch(batch=2, height=64, width=96, frame_ids=frame_ids, seed=62, depth_hints=True)
    _check(pb, dev, True, {}, want_T=True)


@pytest.mark.parametrize("frame_ids,shape", [((0, -1, 1, "s"), (2, 50, 70)), ((0, "s"), (4, 320, 1024))])
def test_colour_grads_sizes(dev, frame_ids, shape):
    """A ragged size with W % 4 != 0, and the config-4 size 1024x320 (B=4, 4 scales)."""
    B, H, W = shape
    scales = (0, 1, 2, 3) if H % 8 == 0 and W % 8 == 0 else (0, 1)
    pb = synth.photo_batch(batch=B, height=H, width=W, frame_ids=frame_ids, scales=scales, seed=63, depth_hints=True)
    _check(pb, dev, True, {})


@pytest.mark.parametrize("frame_ids", [(0, "s"), (0, -1, 1, "s")])
def test_colour_grads_per_scale_upstream(dev, frame_ids):
    """Distinct upstream weights on `loss` and on every `loss/s`, `reproj_loss/s` and `depth_hint_loss/s`."""
    pb = synth.photo_batch(batch=2, height=64, width=96, frame_ids=frame_ids, seed=64, depth_hints=True)
    up = [0.7, 1.3, -0.4, 2.0, 0.25, 0.9, -1.1, 0.35, 1.6, 0.5, -0.8, 1.2, 0.15]
    _check(pb, dev, True, {}, up=up)


@pytest.mark.parametrize("which", ["target", "source", "pyramid"])
def test_colour_grads_subsets(dev, which):
    """Only one colour input requires grad: it matches the oracle, every other keeps .grad None."""
    pb = synth.photo_batch(batch=2, height=64, width=96, frame_ids=(0, -1, 1, "s"), seed=65, depth_hints=True)
    keys = {"target": [(0, 0)], "source": [(1, 0)], "pyramid": [(0, 2)]}[which]
    _check(pb, dev, True, {}, keys=keys)


def test_colour_grads_full_size_properties(dev):
    """Config 4 (B=8 of 1024x320, [0,'s']): the target and pyramid gradients are bit-identical over two runs (the
    source gradient is scattered atomically: equal to 1e-6 of its maximum); a 3x upstream gives 3x the gradients."""
    pb = synth.photo_batch(batch=8, height=320, width=1024, frame_ids=(0, "s"), seed=66, depth_hints=True)
    keys = _colour_keys(pb)
    a = _run(pb, dev, True, {}, keys, want_sel=False)[4]
    b = _run(pb, dev, True, {}, keys, want_sel=False)[4]
    c = _run(pb, dev, True, {}, keys, up=[3.0] + [0.0] * (3 * len(pb.scales)), want_sel=False)[4]
    for k in keys:
        if k[0] == 0:
            assert torch.equal(a[k], b[k]), k
        else:
            assert_close(b[k], a[k], 1e-6, "source %s rerun" % (k,))
        assert float(a[k].abs().max()) > 0, k
        assert_close(c[k], 3.0 * a[k], TOL, "3x upstream %s" % (k,))


def test_colour_grads_cuda_graph_replay(dev):
    """Forward + backward (colour and disparity gradients) captured in a CUDA graph and replayed equals eager."""
    pb = synth.photo_batch(batch=2, height=64, width=96, frame_ids=(0, -1, 1, "s"), seed=67, depth_hints=True)
    g = pb.to(dev)
    keys = _colour_keys(pb)
    colors = {k: v.clone().requires_grad_(k in keys) for k, v in g.color.items()}
    disps = {s: v.clone().requires_grad_(True) for s, v in g.disp.items()}
    noise = {s: g.noise[s][:, :1].contiguous() for s in g.scales}
    ins = [colors[k] for k in keys] + [disps[s] for s in g.scales]

    def run():
        losses, _ = DH.depth_hint_losses(colors, disps, g.K, g.inv_K, g.T, g.frame_ids, g.scales, g.height, g.width,
                                         g.extras["depth_hint"], g.extras["depth_hint_mask"], True, noise=noise)
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
        assert float(e.abs().max()) > 0, i
        assert_close(r, e, 1e-6, "graph replay input %d" % i)


def test_colour_grads_bf16_frames(dev):
    """bf16 frames: the gradients come back in bf16, within the bf16 class of the oracle on the rounded frames."""
    pb = synth.photo_batch(batch=2, height=64, width=96, frame_ids=(0, -1, 1, "s"), seed=68, depth_hints=True)
    for k in list(pb.color):
        pb.color[k] = pb.color[k].to(torch.bfloat16).float()
    keys = _colour_keys(pb)
    gc = _run(pb, dev, True, {}, keys, dtype=torch.bfloat16)[4]
    ref32 = _oracle(pb, True, {}, torch.float32, keys)
    ref64 = _oracle(pb, True, {}, torch.float64, keys)
    for k in keys:
        assert gc[k].dtype == torch.bfloat16, k
        assert_grad_close(gc[k].float(), ref32[k], ref64[k], 4e-3, "bf16 grad colour %s" % (k,), outlier_frac=OUTL)


def test_dh_compute_losses_colour_grads(dev):
    """The patched depth-hints Trainer.compute_losses on a namespace trainer: inputs[("color", f, s)] requiring grad
    receive the oracle's gradients."""
    pb = synth.photo_batch(batch=2, height=64, width=96, frame_ids=(0, -1, "s"), seed=69, depth_hints=True)
    g = pb.to(dev)
    opt = types.SimpleNamespace(v1_multiscale=False, pose_model_type="separate_resnet", predictive_mask=False,
                                adv_train=False, scales=list(g.scales), frame_ids=list(g.frame_ids), height=g.height,
                                width=g.width, min_depth=pb.min_depth, max_depth=pb.max_depth, use_depth_hints=True,
                                no_ssim=False, avg_reprojection=False, disable_automasking=False,
                                disparity_smoothness=1e-3)
    trainer = types.SimpleNamespace(opt=opt, _dmh_noise={s: g.noise[s][:, :1].contiguous() for s in g.scales})
    inputs = {("color", f, s): v.clone().requires_grad_(True) for (f, s), v in g.color.items()}
    inputs[("K", 0)], inputs[("inv_K", 0)], inputs["stereo_T"] = g.K, g.inv_K, g.T["s"]
    inputs["depth_hint"], inputs["depth_hint_mask"] = g.extras["depth_hint"], g.extras["depth_hint_mask"]
    outputs = {("disp", s): g.disp[s].clone().requires_grad_(True) for s in g.scales}
    outputs[("cam_T_cam", 0, -1)] = g.T[-1]
    losses = DH.dh_compute_losses(trainer, inputs, outputs)
    losses["loss"].backward()
    keys = _colour_keys(pb)
    ref32 = _oracle(pb, True, {}, torch.float32, keys)
    ref64 = _oracle(pb, True, {}, torch.float64, keys)
    for (f, s) in keys:
        assert_grad_close(inputs[("color", f, s)].grad, ref32[(f, s)], ref64[(f, s)], TOL, "color %s %s" % (f, s),
                          outlier_frac=OUTL)


# ---------------------------------------------------------------------- winning-source bits of dmh_photo_scale_dh
def _photo_scale_dh(g, s, hints, over, flags):
    """One dmh_photo_scale_dh launch for scale s, set up as depth_hints._ObjectiveDH does (planar sources)."""
    lib = _lib.load()
    ids, srcs, target, B, hint_rl, _, ident = DH._prologue(
        g.color, g.T, g.frame_ids, g.height, g.width, g.extras["depth_hint"], g.extras["depth_hint_mask"], hints,
        False, False, g.K, g.inv_K)
    H, W = g.height, g.width
    d = g.disp[s]
    dev = target.device
    part = torch.empty(4, B * lib.dmh_photo_tiles(H, W), device=dev)
    g_r = torch.empty(B, 1, H, W, device=dev)
    g_h = torch.empty(B, 1, H, W, device=dev) if hints else None
    sel = torch.empty(B, H, W, device=dev, dtype=torch.uint8)
    hd, hv = (g.extras["depth_hint"], g.extras["depth_hint_mask"]) if hints else (None, None)
    noise = g.noise[s][:, :1].contiguous()      # held until the launch: a copy made in the argument list is freed early
    Ts = [g.T[f] for f in ids]
    if over.get("avg_reprojection"):
        flags |= ops.FLAG_AVG_REPROJECTION
    check(lib.dmh_photo_scale_dh(ptr(target), ptr_array(srcs), ptr_array(Ts), len(srcs), ptr(d), d.shape[2],
                                 d.shape[3], ptr(g.K), ptr(g.inv_K), ptr(ident), ptr(noise), ptr(hint_rl), ptr(hd),
                                 ptr(hv), B, H, W, g.min_depth, g.max_depth, flags, ptr(part), ptr(g_r), ptr(g_h), None,
                                 ptr(sel), stream()), "photo_scale_dh")
    torch.cuda.synchronize()
    return sel.cpu(), [t.cpu() for t in (part, g_r, g_h) if t is not None]


def _oracle_first_min(pb, s):
    """fp64 oracle: the source frame whose reprojection loss is the (first) minimum, and the gap to the runner-up"""
    dt = torch.float64
    disp = F.interpolate(pb.disp[s].to(dt), [pb.height, pb.width], mode="bilinear", align_corners=False)
    rl = []
    for f in pb.frame_ids[1:]:
        pred, _, _ = OP.warp_from_disp(disp, pb.color[(f, 0)].to(dt), pb.K.to(dt), pb.inv_K.to(dt), pb.T[f].to(dt),
                                       pb.min_depth, pb.max_depth)
        rl.append(OP.reprojection_loss(pred, pb.color[(0, 0)].to(dt), False))
    rl = torch.cat(rl, 1)
    idx = torch.min(rl, dim=1)[1]
    srt = rl.sort(1).values
    return idx, srt[:, 1] - srt[:, 0]


@pytest.mark.parametrize("frame_ids,hints,over", [((0, -1, 1, "s"), True, {}), ((0, -1, 1), False, {}),
                                                  ((0, "s"), True, {}),
                                                  ((0, -1, "s"), True, dict(avg_reprojection=True))])
def test_sel_source_bits(dev, frame_ids, hints, over):
    """With DMH_PHOTO_SEL_SOURCE: sel & 3 equals the unflagged sel bit for bit and the sums / gradients are unchanged;
    sel >> 2 is the oracle's first-minimum source wherever the sources are not within 1e-5 of each other, and 0 with
    one source (the fast kernel) or under avg_reprojection."""
    pb = synth.photo_batch(batch=2, height=64, width=96, frame_ids=frame_ids, seed=70, depth_hints=True)
    g = pb.to(dev)
    multi = len(frame_ids) > 2 and not over.get("avg_reprojection")
    for s in (0, 2):
        sel0, outs0 = _photo_scale_dh(g, s, hints, over, 0)
        sel1, outs1 = _photo_scale_dh(g, s, hints, over, ops.FLAG_SEL_SOURCE)
        assert torch.equal(sel1 & 3, sel0), s
        assert int(sel0.max()) <= 2, s
        for a, b in zip(outs1, outs0):
            assert torch.equal(a, b), s
        src = (sel1 >> 2).long()
        if not multi:
            assert int(src.max()) == 0, s
            continue
        idx, gap = _oracle_first_min(pb, s)
        clear = gap > 1e-5
        assert float(clear.float().mean()) > 0.95, s
        assert torch.equal(src[clear], idx[clear]), s
        assert int(src.max()) == len(frame_ids) - 2, s          # every source wins somewhere
