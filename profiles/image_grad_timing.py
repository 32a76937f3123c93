#!/usr/bin/env python
"""Forward + backward of the fused objective with and without the colour-frame gradients (CUDA events), and the
kernel times of the colour-gradient launches, for BASELINE config 2 (B=32, 1024x320, [0,'s'], 4 scales),
mono+stereo (B=32, 1024x320, [0,-1,1,'s'], pose gradients) and the depth-hints objective of BASELINE config 4
(B=32, 1024x320, [0,'s'], 4 scales, depth_hints.depth_hint_losses).  Also the CUDA-graph replay of
objective.GraphedObjective at BASELINE config 1 size (B=4, 640x192, [0,'s'], 4 scales) without gradients for the
frames and the pose, with the frames' and with both, and ops.photo_scale_sum forward + backward (one scale,
B=32, 1024x320, [0,'s'], identity candidates) without and with the target, source and identity gradients.  The runs
without and with colour gradients alternate.  Prints the card and its power limit with the numbers.
usage: python profiles/image_grad_timing.py [--iters 20] [--batch 32]"""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from depthmodelhardening_b200 import depth_hints, objective, ops, synth  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "nvidia-smi unavailable"
    return "%s | %s" % (torch.cuda.get_device_name(0), q)


def bytes_per_px(F, S):
    """Algorithmic bytes per target pixel of the colour-gradient launches (fp32): S reprojection launches and one
    identity launch (none for the depth-hints objective).  Per scale: read 12 target + 12 F gathered sources + <= 4
    disparity + 1 sel, write 24 target read-modify-write + 12 F source RED; identity: read 12 + 12 F + S sel, write
    12 + 12 F."""
    return S * (12 + 12 * F + 4 + 1 + 24 + 12 * F), (12 + 12 * F + S) + (12 + 12 * F)


def timed_loop(fn, iters, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def run_case(name, frame_ids, B, H, W, iters, dev, hints=False):
    pb = synth.photo_batch(batch=B, height=H, width=W, frame_ids=frame_ids, seed=5, depth_hints=hints).to(dev)
    F = len(frame_ids) - 1
    S = len(pb.scales)
    noise1 = {s: pb.noise[s][:, :1].contiguous() for s in pb.scales}

    def make(colour):
        colors = {k: v.clone().requires_grad_(colour) for k, v in pb.color.items()}
        disps = {s: v.clone().requires_grad_(True) for s, v in pb.disp.items()}
        Ts = {k: v.clone().requires_grad_(k != "s") for k, v in pb.T.items()}

        def step():
            if hints:
                losses, _ = depth_hints.depth_hint_losses(colors, disps, pb.K, pb.inv_K, Ts, pb.frame_ids, pb.scales, H,
                                                          W, pb.extras["depth_hint"], pb.extras["depth_hint_mask"], True,
                                                          noise=noise1)
            else:
                losses, _ = objective.photometric_losses(colors, disps, pb.K, pb.inv_K, Ts, pb.frame_ids, pb.scales, H,
                                                         W, noise=pb.noise)
            losses["loss"].backward()
        return step

    base, with_c = make(False), make(True)
    t0 = timed_loop(base, iters)
    t1 = timed_loop(with_c, iters)
    t0b = timed_loop(base, iters)                  # alternate: the spread of the baseline shows in t0 vs t0b
    t1b = timed_loop(with_c, iters)
    ops.KERNEL_EVENTS = []
    for _ in range(iters):
        with_c()
    torch.cuda.synchronize()
    per = {}
    for n, a, b in ops.KERNEL_EVENTS:
        if n in ("identity_image_grad", "photo_image_grad", "photo_image_grad_dh"):
            per.setdefault(n, []).append(a.elapsed_time(b))
    ops.KERNEL_EVENTS = None
    print("%s: B=%d %dx%d frames=%s scales=%d" % (name, B, W, H, list(frame_ids), S))
    print("  fwd+bwd without colour grads  %.3f ms / %.3f ms (two runs)" % (t0, t0b))
    print("  fwd+bwd with colour grads     %.3f ms / %.3f ms (two runs)" % (t1, t1b))
    npx = B * H * W
    per_scale_b, ident_b = bytes_per_px(F, S)
    for n, ts in sorted(per.items()):
        ts = sorted(ts)
        med = ts[len(ts) // 2]
        nbytes = (ident_b if n == "identity_image_grad" else per_scale_b / S) * npx
        print("  %-20s median %.3f ms per launch (%d launches), %.0f B/px algorithmic -> %.2f TB/s" % (
            n, med, len(ts), nbytes / npx, nbytes / med / 1e9))


def run_graphed(B, H, W, iters, dev):
    """GraphedObjective replay: disparity gradients only, plus every frame's, plus the stereo pose's"""
    pb = synth.photo_batch(batch=B, height=H, width=W, frame_ids=(0, "s"), seed=5).to(dev)
    variants = [("disparities only", False, False), ("+ frames", True, False), ("+ frames + pose", True, True)]
    graphs = []
    for name, cols, pose in variants:
        colors = {k: v.clone().requires_grad_(cols) for k, v in pb.color.items()}
        Ts = {k: v.clone().requires_grad_(pose) for k, v in pb.T.items()}
        graphs.append((name, objective.GraphedObjective(colors, pb.disp, pb.K, pb.inv_K, Ts, pb.frame_ids, pb.scales, H,
                                                        W, noise=pb.noise)))
    print("GraphedObjective replay (config 1 size): B=%d %dx%d frames=[0, 's'] scales=%d" % (B, W, H, len(pb.scales)))
    times = {name: [] for name, _ in graphs}
    for _ in range(2):                             # alternate the variants: the spread shows in the two runs
        for name, g in graphs:
            times[name].append(timed_loop(g, iters))
    for name, _ in graphs:
        print("  replay, %-18s %.3f ms / %.3f ms (two runs)" % (name, *times[name]))


def run_scale_sum(B, H, W, iters, dev):
    """ops.photo_scale_sum forward + backward at full resolution, without and with the input gradients"""
    pb = synth.photo_batch(batch=B, height=H, width=W, frame_ids=(0, "s"), scales=(0,), seed=5).to(dev)
    target, src = pb.color[(0, 0)], pb.color[("s", 0)]
    ident = torch.empty(B, 1, H, W, device=dev)
    from depthmodelhardening_b200._lib import check, ptr, ptr_array, stream
    check(ops._lib_().dmh_identity_loss(ptr(target), ptr_array([src]), 1, B, H, W, 0, ptr(ident), stream()),
          "identity_loss")

    def make(grads):
        tg, sr, idn = (t.clone().requires_grad_(grads) for t in (target, src, ident))
        d = pb.disp[0].clone().requires_grad_(True)

        def step():
            total, _ = ops.photo_scale_sum(d, tg, [sr], [pb.T["s"]], pb.K, pb.inv_K, ident=idn, noise=pb.noise[0])
            total.backward()
        return step

    base, with_g = make(False), make(True)
    t = [timed_loop(base, iters), timed_loop(with_g, iters), timed_loop(base, iters), timed_loop(with_g, iters)]
    print("photo_scale_sum: B=%d %dx%d frames=[0, 's'], one scale" % (B, W, H))
    print("  fwd+bwd without frame / identity grads  %.3f ms / %.3f ms (two runs)" % (t[0], t[2]))
    print("  fwd+bwd with frame / identity grads     %.3f ms / %.3f ms (two runs)" % (t[1], t[3]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--batch", type=int, default=32)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("image_grad_timing.py needs a CUDA device")
    dev = torch.device("cuda:0")
    print(card())
    run_case("config 2", (0, "s"), a.batch, 320, 1024, a.iters, dev)
    run_case("mono+stereo", (0, -1, 1, "s"), a.batch, 320, 1024, a.iters, dev)
    run_case("config 4 (depth hints)", (0, "s"), a.batch, 320, 1024, a.iters, dev, hints=True)
    run_graphed(4, 192, 640, max(a.iters, 200), dev)
    run_scale_sum(a.batch, 320, 1024, a.iters, dev)


if __name__ == "__main__":
    main()
