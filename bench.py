#!/usr/bin/env python
"""bench.py -- hot-path benchmark (contract: see task statement / DESIGN.md).

One "step" = one pass of the grafted hot path over one batch of synthetic input:
  stage 1  physical-patch PGD step: patch-apply fwd (perspective warp + composite
           + anti-aliased resize) -> patch-apply bwd from a supplied upstream
           gradient -> [allreduce of the shared patch gradient when N>1] -> L-inf
           sign/project update                          (Ba = per-GPU batch)
  stage 2  monodepth2 photometric objective fwd+bwd: 4 scales, automask, SSIM+L1,
           smoothness, gradients w.r.t. the 4 disparity maps   (B = per-GPU batch)
Workload = BASELINE.json configs[1]: 1024x320, batch 32 per GPU, frame_ids [0,'s'].
The depth network is outside the graft and is not part of the step.

metric  reproj-loss fwd+bwd Mpix/s (target pixels N*B*H*W per step / step time);
        PGD steps/s and the per-stage split are reported in extra keys.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

H, W = 320, 1024
SCALES = (0, 1, 2, 3)
FRAME_IDS = (0, "s")
GLOBAL_BATCH = 32           # north_star: batch 32 sharded across the GPUs (strong-scaling sub-record)
METRIC = "reproj_loss_fwd_bwd_mpix_per_s"
UNIT = "Mpix/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40,
                    help="timed steps of the headline and of the per-stage split; the informational sub-records keep "
                         "their own counts: strong scaling max(steps, 20), end to end max(4, steps // 2), multi-source "
                         "max(5, steps // 2), eager reference on the GPU 6")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=32, help="per-GPU batch (weak scaling)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-e2e-u8", action="store_true",
                    help="skip the additional (informational) end-to-end measurement with 8-bit frame transport")
    ap.add_argument("--no-e2e-bf16", action="store_true",
                    help="skip the additional (informational) end-to-end measurement with bf16 frame transport")
    ap.add_argument("--no-patch", action="store_true", help="skip stage 1 (debug)")
    ap.add_argument("--attack", default="l0", choices=["l0", "linf"],
                    help="stage-1 update rule: l0 = README config (--norm_type l_0), linf = sign/project step")
    ap.add_argument("--cpu-sample-batch", type=int, default=0,
                    help="batch slice of the CPU legs (0: cpu_baseline 8; --impl reference: adaptive, see reference_arm)")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling (sharded batch 32) sub-record")
    ap.add_argument("--no-gpu-eager", action="store_true", help="skip the reference-on-the-same-GPU baseline")
    ap.add_argument("--strong-shard", type=int, default=0,
                    help="N = 1 only: also time the step at the shard size of a K-GPU strong-scaling run (batch 32 / K "
                         "items, no collective) -- sub-record strong_shard_emulation")
    ap.add_argument("--no-graph", action="store_true",
                    help="headline = the step launched from Python on one stream (default: CUDA-graph replay, two streams)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu_index = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(prefix="dmh_clocks_", suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1]))
                    mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            sm.sort()
            out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


# ----------------------------------------------------------------------------- workload
def make_host_workload(batch, rank, with_patch):
    from depthmodelhardening_b200 import synth
    pb = synth.photo_batch(batch=batch, height=H, width=W, frame_ids=FRAME_IDS, scales=SCALES, seed=1000 * rank)
    pt = synth.patch_batch(batch=batch, seed=1000 * rank) if with_patch else None
    return pb, pt


def algorithmic_bytes(batch, F=1, S=4):
    """SURVEY.md 8(d) compulsory traffic (fp32)."""
    sigma = sum(4.0 ** (-s) for s in range(S))
    fwd = 12 + 12 * F + 4 * S + 4 * F * S + (4 * sigma + 12 * (sigma - 1))
    bwd = fwd + 4 * S + 4 * sigma
    per_px = fwd + bwd
    return per_px * batch * H * W, per_px


class Stage2:
    def __init__(self, pb, device, noise_mode="injected"):
        self.g = pb.to(device)
        self.noise_mode = noise_mode
        self.disps = {s: self.g.disp[s].clone().requires_grad_(True) for s in self.g.scales}

    def step(self):
        from depthmodelhardening_b200 import objective
        g = self.g
        for d in self.disps.values():
            d.grad = None
        losses, _ = objective.photometric_losses(
            g.color, self.disps, g.K, g.inv_K, g.T, g.frame_ids, g.scales, g.height, g.width,
            noise=g.noise if self.noise_mode == "injected" else None,
            noise_mode="device" if self.noise_mode != "injected" else "reference")
        losses["loss"].backward()
        # what a caller of the objective receives: the losses and the disparity gradients.  Detached: a loss kept with
        # its grad_fn keeps this step's autograd graph alive, and the next CUDA-graph capture then fails on the stale
        # AccumulateGrad nodes
        self.outputs = {k.replace("/", "_"): v.detach() for k, v in losses.items()}
        self.outputs.update({"grad_disp_%d" % s: d.grad for s, d in self.disps.items()})
        return losses["loss"]


class Stage1:
    """One PGD iteration of the physical patch attack with the depth network's gradient supplied
    (the network is outside the graft): [L0: compose patterns + count] -> patch apply fwd -> bwd to the
    patch -> [all-reduce] -> update (L0: mask-cost gradient + Adam, README `--norm_type l_0`; or L-inf)."""

    def __init__(self, pt, device, world, attack="l0"):
        import numpy as np
        from depthmodelhardening_b200 import patch_ops, synth
        self.ops = patch_ops
        self.g = pt.to(device)
        P34 = np.array(patch_ops.KITTI_P2_003086, dtype=np.float64).reshape(3, 4)
        self.coeffs = patch_ops.homographies(pt.z0, pt.alpha, P34, obj_hw=(synth.PATCH_H, synth.PATCH_W)).to(device)
        self.adv = self.g.obj.clone()
        self.world = world
        self.attack = attack
        self.gbuf = None
        # the step's one collective: one kernel over NVLink peer memory (dist.PeerReducer, csrc/peer_reduce.cu) when
        # symmetric memory is available; DMH_PEER_REDUCE=0 (or no peer access) keeps the NCCL all-reduce + scaling
        self.peer = None
        if world > 1 and os.environ.get("DMH_PEER_REDUCE", "1") != "0":
            from depthmodelhardening_b200 import dist as D
            if D.PeerReducer.available():
                self.peer = D.PeerReducer(self.adv.numel() + 1, device)
        if attack == "l0":      # M2/trainer.py:216-218: adam_lr 0.5, mask_wt 0.06, l0_thresh 0.1
            self.l0 = patch_ops.L0State(self.g.obj, self.g.pattern_pos, self.g.pattern_neg, lr=0.5, betas=(0.5, 0.9))
            self.first = True

    def step(self):
        ops = self.ops
        g = self.g
        if self.attack == "l0":
            self.adv = self.l0.compose_count(first=self.first)
            self.first = False
        if self.peer is not None:
            # the ONE collective of the step, without NCCL: the backward kernel accumulates into the rank's symmetric
            # buffer, one kernel sums all ranks' buffers over NVLink in rank order, averages, and (L-inf) updates
            adv_scene, mask_out, _ = ops.apply_patch_fwd_bwd(self.adv, g.mask, g.scenes, self.coeffs, g.upstream,
                                                             grad_out=self.peer.buffer)
            if self.attack != "l0":
                new_adv = torch.empty_like(self.adv)
                self.peer.allreduce(average=True, linf=(self.adv, g.obj, 0.02, 0.1, new_adv))
                self.outputs = {"adv_scene": adv_scene, "mask": mask_out, "patch": self.adv, "patch_next": new_adv}
                self.adv = new_adv
                return adv_scene
            grad_patch = self.peer.allreduce(average=True)[:self.adv.numel()].view_as(self.adv)
        elif self.world > 1:
            # the ONE collective of the step: the backward kernel writes the patch gradient straight into the
            # all-reduce buffer (the scalar attack loss rides in its last element); all-reduce in place
            if self.gbuf is None:
                self.gbuf = torch.zeros(self.adv.numel() + 1, device=self.adv.device)
            adv_scene, mask_out, grad_patch = ops.apply_patch_fwd_bwd(self.adv, g.mask, g.scenes, self.coeffs, g.upstream,
                                                                      grad_out=self.gbuf)
            torch.distributed.all_reduce(self.gbuf)
            self.gbuf.div_(self.world)
        else:
            adv_scene, mask_out, grad_patch = ops.apply_patch_fwd_bwd(self.adv, g.mask, g.scenes, self.coeffs, g.upstream)
        # what a caller of the step receives: the patched scenes, the resized mask, the patch gradient, the patch the
        # step applied and the updated attack state
        self.outputs = {"adv_scene": adv_scene, "mask": mask_out, "grad_patch": grad_patch, "patch": self.adv}
        if self.attack == "l0":
            self.l0.adam_step(grad_patch, 0.06, 0.1)
            self.outputs.update(pattern_pos=self.l0.ppos, pattern_neg=self.l0.pneg)
        else:
            self.adv = ops.pgd_linf_step(self.adv, grad_patch, g.obj, alpha=0.02, eps=0.1)
            self.outputs["patch_next"] = self.adv
        return adv_scene


def timed_loop(fn, steps, warmup, world):
    for _ in range(warmup):
        fn()
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms = float(t.item())
        torch.distributed.barrier()
    return ms / steps


DUMP_MAX_ELEMENTS = 1 << 21     # per array (8 MB of fp32): at the default workload the whole dump is ~40 MB
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(outputs, out_dir):
    """Writes every output as out_dir/<name>.npy in float32.  An array with more than DUMP_MAX_ELEMENTS elements is
    replaced by a fixed sample of its flattened elements: DUMP_MAX_ELEMENTS seeded draws of an index, duplicates
    dropped, in index order -- the same indices in every run, so that the dumps of two builds compare element for
    element.  The objective's outputs repeat bit for bit; the patch gradient
    is summed in no fixed order, so the attack state (patch, pattern_*) differs between two runs of the same build by
    that rounding, amplified by every Adam iteration before the last timed step."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, t in sorted(outputs.items()):
        flat = t.detach().float().reshape(-1)
        if flat.numel() > DUMP_MAX_ELEMENTS:
            idx = np.sort(np.random.default_rng(0).integers(0, flat.numel(), DUMP_MAX_ELEMENTS))
            idx = idx[np.concatenate(([True], idx[1:] != idx[:-1]))]
            flat = flat[torch.from_numpy(idx).to(flat.device)]
            a = flat.cpu().numpy()
        else:
            a = flat.cpu().numpy().reshape(tuple(t.shape))
        total += a.nbytes
        if total > DUMP_MAX_BYTES:
            raise RuntimeError("--dump-outputs: more than %d bytes" % DUMP_MAX_BYTES)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def stage1_stream(device):
    """The side stream stage 1 runs on beside stage 2 (DMH_S1_PRIORITY, default 0 = the priority of stage 2's stream).
    Measured on one box (profiles/r02_kernel_ab.txt, block r3a): a high-priority stage-1 stream is SLOWER -- 1.877 vs
    1.866 ms at 32 items, 0.2845 vs 0.2753 ms at 4 items per GPU: stage 1's short kernels then displace CTAs of the
    photometric kernel, which is the critical path, instead of filling its tail."""
    return torch.cuda.Stream(device=device, priority=int(os.environ.get("DMH_S1_PRIORITY", "0")))


def capture_step(s1, s2, device, lib, two_stream=True):
    """One step (stage 1 incl. its collective, stage 2 fwd+bwd) captured into a CUDA graph; returns (graph, number of
    this library's kernel launches inside one replay).  two_stream: stage 1 runs on a side stream beside stage 2."""
    cur = torch.cuda.current_stream()
    side = stage1_stream(device)
    side.wait_stream(cur)
    with torch.cuda.stream(side):                          # warm-up off the capturing stream (allocator, lazy inits)
        for _ in range(3):
            s1.step()
            s2.step()
    cur.wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    n0 = lib.dmh_launch_count()
    with torch.cuda.graph(graph):
        if two_stream:
            cs = torch.cuda.current_stream()
            side.wait_stream(cs)
            with torch.cuda.stream(side):
                s1.step()
            s2.step()
            cs.wait_stream(side)
        else:
            s1.step()
            s2.step()
    return graph, int(lib.dmh_launch_count() - n0)


def measure_strong(args, rank, world, device, global_batch, shard=1):
    """Strong scaling (north_star / SURVEY.md 8(e)): the batch-32 step with the batch SHARDED over the ranks.
    Same step as the headline (stage 1 + the one all-reduce + stage 2); timed eagerly and as a CUDA-graph replay of
    the whole step (the all-reduce included): with 4 items per GPU the eager step is launch-bound.
    shard > 1 (world == 1): emulate the shard of a `shard`-GPU run on this GPU (no collective)."""
    if global_batch % (world * shard) != 0:
        return {"error": "global batch %d not divisible by %d ranks" % (global_batch, world * shard)}
    Bs = global_batch // (world * shard)
    pb, pt = make_host_workload(Bs, rank, True)
    s2 = Stage2(pb, device)
    s1 = Stage1(pt, device, world, args.attack)

    def step():
        s1.step()
        return s2.step()

    steps = max(args.steps, 20)
    ms_eager = timed_loop(step, steps, max(args.warmup, 3), world)
    out = {"global_batch": global_batch, "per_gpu_batch": Bs, "n_gpus": world, "ms_per_step_eager": ms_eager,
           "value_eager": global_batch * H * W / (ms_eager * 1e-3) / 1e6, "unit": UNIT, "scaling": "strong"}
    cur = torch.cuda.current_stream()
    side = stage1_stream(device)
    side.wait_stream(cur)
    with torch.cuda.stream(side):
        for _ in range(3):
            step()
    cur.wait_stream(side)
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    ms_graph = timed_loop(graph.replay, steps, max(args.warmup, 3), world)
    # informational: the two stages of a step read different inputs (stage 1 of step i+1 does not depend on stage 2
    # of step i: a trainer can pipeline them), so a second capture runs stage 1 -- with its all-reduce -- on a side
    # stream beside stage 2; at 4 items per GPU both are latency-bound chains and overlap almost completely
    try:
        graph2 = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph2):
            cs = torch.cuda.current_stream()
            side.wait_stream(cs)
            with torch.cuda.stream(side):
                s1.step()
            s2.step()
            cs.wait_stream(side)
        ms_graph2 = timed_loop(graph2.replay, steps, max(args.warmup, 3), world)
        out.update({"ms_per_step_two_stream": ms_graph2,
                    "value_two_stream": global_batch * H * W / (ms_graph2 * 1e-3) / 1e6})
    except Exception as exc:
        out["two_stream_error"] = "%s: %s" % (type(exc).__name__, exc)
    out.update({"ms_per_step": ms_graph, "value": global_batch * H * W / (ms_graph * 1e-3) / 1e6,
                "collective": "dmh_peer_allreduce (one kernel over NVLink peer memory)" if s1.peer is not None
                              else ("nccl all_reduce + div_" if world > 1 else "none"),
                "note": "ms_per_step / value: CUDA-graph replay of the whole step (stage 1, the all-reduce of the "
                        "patch gradient, stage 2 fwd+bwd) captured once; *_eager: the same step launched from Python. "
                        "The L0 Adam step index lives on the device (dmh_l0_adam_step_dev): replays are exact."})
    if world > 1:
        # the collective alone, both forms, back to back on this box (device time, max over ranks)
        n = s1.adv.numel() + 1
        buf = torch.zeros(n, device=device)

        def nccl():
            torch.distributed.all_reduce(buf)
            buf.div_(world)
        us = {"nccl_all_reduce_plus_div": 1e3 * timed_loop(nccl, 200, 20, world)}
        if s1.peer is not None:
            us["peer_memory_kernel"] = 1e3 * timed_loop(lambda: s1.peer.allreduce(average=True), 200, 20, world)
        out["allreduce_us"] = us
    return out


def measure_multisource(args, device, batch):
    """Informational (N = 1): the objective of configs[1] read as TRUE mono+stereo (SURVEY.md 8(d): F = 3,
    frame_ids [0,-1,1,'s'], pose gradients for the temporal frames) and BASELINE configs[4] (two temporal sources,
    batch 16), each through the multi-source tile kernel (csrc/photo_mf.cu, one launch for all sources and scales)
    and through the general per-scale kernel it replaces."""
    from depthmodelhardening_b200 import objective, ops, synth
    out = {}
    for key, B_, fids in (("mono_stereo_f3", batch, (0, -1, 1, "s")), ("multi_frame_f2_b16", 16, (0, -1, 1))):
        pb = synth.photo_batch(batch=B_, height=H, width=W, frame_ids=fids, scales=SCALES, seed=6).to(device)
        disps = {s_: pb.disp[s_].clone().requires_grad_(True) for s_ in pb.scales}
        Ts = {k: v.clone().requires_grad_(k != "s") for k, v in pb.T.items()}

        def step():
            for d in disps.values():
                d.grad = None
            for t in Ts.values():
                t.grad = None
            losses, _ = objective.photometric_losses(pb.color, disps, pb.K, pb.inv_K, Ts, pb.frame_ids, pb.scales, H, W,
                                                     noise=pb.noise)
            losses["loss"].backward()
        rec = {"per_gpu_batch": B_, "frame_ids": [str(f) for f in fids], "unit": UNIT}
        for name, flag in (("tile_kernel", True), ("general_kernel", False)):
            old = ops.MULTISOURCE
            ops.MULTISOURCE = flag
            try:
                ms = timed_loop(step, max(5, args.steps // 2), 3, 1)
            finally:
                ops.MULTISOURCE = old
            rec["ms_per_step_" + name] = ms
            rec["value_" + name] = B_ * H * W / (ms * 1e-3) / 1e6
        out[key] = rec
        del pb, disps, Ts
        torch.cuda.empty_cache()
    out["note"] = ("stage 2 only (objective fwd+bwd incl. pose gradients); tile_kernel = dmh_photo_multisource "
                   "(photo_mf_kernel: all sources and scales in one launch), general_kernel = dmh_photo_scale per scale "
                   "(photo_scale_kernel<F>, the round-1 path)")
    return out


# ----------------------------------------------------------------------------- CPU baseline / reference arm
def reference_available():
    """The unmodified reference: /root/reference in the build container, else the copy that build() placed under
    oracle/_ref/ (git-ignored, travels to the GPU box with the snapshot)."""
    try:
        from oracle import refload
        return refload.available()
    except Exception:
        return False


def reference_step(sample_batch, with_patch, device="cpu", attack="l0", seed=7):
    """One step of the hot path executed by the REFERENCE'S OWN CODE (oracle/ref_step.py: Trainer.generate_images_pred
    + compute_losses + backward; the L0 PGD iteration on the reference's PhysicalTrans) on `device`."""
    from depthmodelhardening_b200 import synth
    from oracle import ref_step
    pb = synth.photo_batch(batch=sample_batch, height=H, width=W, frame_ids=FRAME_IDS, scales=SCALES, seed=seed)
    pt = synth.patch_batch(batch=sample_batch, seed=seed) if with_patch else None
    if device != "cpu":
        pb = pb.to(device)
        pt = pt.to(device) if pt is not None else None
    s2 = ref_step.Stage2Reference(pb, device)
    s1 = ref_step.Stage1Reference(pt, device) if pt is not None else None

    def step():
        if s1 is not None:
            s1.step()
        return s2.step()["loss"]
    return step


def cpu_port_step(sample_batch, with_patch, attack="l0"):
    """Fallback when the reference copy is absent: the oracle restatement (kind "port")."""
    import numpy as np
    from depthmodelhardening_b200 import synth
    from oracle import patch as OQ
    from oracle import photometric as OP
    from oracle.refload import CALIB_P2
    pb = synth.photo_batch(batch=sample_batch, height=H, width=W, frame_ids=FRAME_IDS, scales=SCALES, seed=7)
    pt = synth.patch_batch(batch=sample_batch, seed=7) if with_patch else None
    P34 = np.array(CALIB_P2, dtype=np.float64).reshape(3, 4)
    state = {}
    if pt is not None:
        state["pp"] = pt.pattern_pos.clone().requires_grad_(True)
        state["pn"] = pt.pattern_neg.clone().requires_grad_(True)
        state["opt"] = torch.optim.Adam([state["pp"], state["pn"]], lr=0.5, betas=(0.5, 0.9))

    def step():
        if pt is not None:
            adv, pos, neg = OQ.l0_compose(pt.obj, state["pp"], state["pn"])
            OQ.l0_count(pos, neg)
            scene, _ = OQ.apply_patch(adv, pt.mask, pt.scenes, pt.z0, pt.alpha, P34)
            cost = (scene * pt.upstream).sum() + 0.06 * OQ.l0_mask_cost(state["pp"], state["pn"])
            state["opt"].zero_grad()
            cost.backward()
            state["opt"].step()
        OP.objective_from_batch(pb)
    return step


def cpu_step_factory(with_patch, attack):
    """(make_step(batch), kind)"""
    if reference_available():
        return (lambda nb: reference_step(nb, with_patch, "cpu", attack)), "reference"
    return (lambda nb: cpu_port_step(nb, with_patch, attack)), "port"


def run_cpu_baseline(sample_batch, with_patch, reps=6, attack="l0"):
    torch.set_num_threads(os.cpu_count() or 1)
    make, kind = cpu_step_factory(with_patch, attack)
    step = make(sample_batch)
    step()
    t0 = time.perf_counter()
    for _ in range(reps):
        step()
    dt = (time.perf_counter() - t0) / reps
    what = ("the reference's own code (oracle/_ref copy: Trainer.generate_images_pred + compute_losses + backward; L0 "
            "PGD iteration on its PhysicalTrans)" if kind == "reference" else "oracle port (torch-CPU restatement)")
    return {"value": sample_batch * H * W / dt / 1e6, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind,
            "sample": "%s on a batch-%d slice of the 1024x320 workload, %d reps after 1 warm-up, %.2f s/step"
                      % (what, sample_batch, reps, dt)}


def reference_arm(args, rank, world):
    """`--impl reference`: the reference's own CPU implementation of the step on the box's host cores, with every
    host thread, on this arm's config / metric / unit.  --steps / --warmup are honoured; the per-step sample is the
    largest batch (<= the per-GPU batch) for which the whole run is projected to end within ~4 minutes."""
    if rank != 0:
        return
    torch.set_num_threads(os.cpu_count() or 1)
    with_patch = not args.no_patch
    make, kind = cpu_step_factory(with_patch, args.attack)
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    budget_s = float(os.environ.get("DMH_REF_BUDGET_S", "240"))
    sb = args.cpu_sample_batch if args.cpu_sample_batch > 0 else args.batch
    while True:
        step = make(sb)
        t0 = time.perf_counter()
        step()                                             # first call: lazy initialisation + a first timing
        t1 = time.perf_counter()
        step()
        probe = time.perf_counter() - t1
        if sb <= 1 or probe * (steps + warmup) <= budget_s:
            break
        sb = max(1, sb // 2)
    for _ in range(max(0, warmup - 2)):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    val = sb * H * W / dt / 1e6
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
            "steps": steps, "warmup": warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.attack, with_patch, args.batch, world),
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind,
                             "sample": "batch-%d slice per step (largest power-of-two fraction of the per-GPU batch %d "
                                       "that keeps %d + %d steps within %.0f s on these cores), %.2f s/step"
                                       % (sb, args.batch, steps, warmup, budget_s, dt)},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def workload_config(attack, with_patch, B, world):
    return {"workload": "configs[1]: monodepth2 1024x320 stereo [0,'s'], 4 scales, automask, SSIM+L1, "
                        "smoothness; step = patch PGD step (stage 1, %s update) + photometric loss fwd/bwd (stage 2)" % attack
                        if with_patch else "configs[1] stage 2 only: photometric loss fwd/bwd",
            "per_gpu_batch": B, "global_batch": B * world, "height": H, "width": W, "frame_ids": list(FRAME_IDS),
            "scales": list(SCALES), "l2_policy": "inputs (2x126 MB frames + 168 MB noise) exceed the 126 MB L2"}


def gpu_eager_baseline(B, with_patch, attack, device, steps=6):
    """The reference's own code (stock eager PyTorch: ATen / cuDNN-free elementwise + grid_sample kernels) on the
    SAME B200, same workload: what the graft buys over running the unmodified repository on this GPU."""
    step = reference_step(B, with_patch, device, attack)
    for _ in range(2):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return {"value": B * H * W / (ms * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": ms, "steps": steps, "kind": "reference",
            "what": "the unmodified reference (oracle/_ref copy) on cuda: Trainer.generate_images_pred + compute_losses "
                    "+ backward and one L0 PGD iteration on its PhysicalTrans, per-GPU batch %d, CUDA events" % B}


# ----------------------------------------------------------------------------- main
def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        reference_arm(args, rank, world)
        return
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    # stdout carries exactly one JSON line: anything a library prints on fd 1 meanwhile (NCCL's version banner at
    # communicator creation, ...) is sent to stderr; the line itself goes to the saved descriptor
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=device)
    from depthmodelhardening_b200 import _lib
    lib = _lib.load()
    with_patch = not args.no_patch
    if with_patch:
        try:
            from depthmodelhardening_b200 import patch_ops  # noqa: F401
        except ImportError:
            with_patch = False

    B = args.batch
    pb_host, pt_host = make_host_workload(B, rank, with_patch)
    s2 = Stage2(pb_host, device)
    s1 = Stage1(pt_host, device, world, args.attack) if with_patch else None

    def step():
        if s1 is not None:
            s1.step()
        return s2.step()

    # inputs > L2 (126 MB): colour frames alone are 2 x 126 MB at B=32, so no explicit flush is needed
    # (1) the step launched from Python, one stream (the round-1 / early round-2 headline; kept as `ms_per_step_eager`)
    n0 = lib.dmh_launch_count()
    ms_eager = timed_loop(step, args.steps, args.warmup, world)
    n1 = lib.dmh_launch_count()
    launches = int((n1 - n0) * args.steps / (args.steps + args.warmup))
    # (2) the product schedule and the headline: the SAME step captured once into a CUDA graph -- stage 1 (with the
    # step's one collective) on a side stream beside stage 2, the two stages read different inputs -- and replayed.
    # Nothing is frozen into the capture that a real run would change: the L0 Adam step index lives on the device
    # (dmh_l0_adam_step_dev), the all-reduce's step counter too (dmh_peer_allreduce).  --no-graph, a failed capture
    # or stage 2 alone: the eager step is the headline.
    schedule = "eager, one stream"
    ms_step, graph = ms_eager, None
    sampler = ClockSampler(local_rank)
    if s1 is not None and not args.no_graph:
        try:
            graph, launches_graph = capture_step(s1, s2, device, lib, two_stream=True)
            if world > 1:
                torch.distributed.barrier()
            sampler.start()
            ms_step = timed_loop(graph.replay, args.steps, args.warmup, world)
            launches = launches_graph * args.steps
            schedule = "CUDA-graph replay, stage 1 on a side stream beside stage 2"
        except Exception as exc:
            schedule = "eager, one stream (graph capture failed: %s: %s)" % (type(exc).__name__, str(exc)[:120])
            graph = None
            torch.cuda.synchronize()
    if graph is None:
        sampler.start()
        ms_step = timed_loop(step, args.steps, args.warmup, world)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        # the last timed step's results (a replay rewrites the tensors the capture allocated), before any other
        # measurement below steps the attack state or the objective again
        outputs = dict(s2.outputs)
        if s1 is not None:
            outputs.update(s1.outputs)
        dump_outputs(outputs, args.dump_outputs)

    # per-stage split (same loop, one stage at a time)
    ms_s2 = timed_loop(s2.step, args.steps, 2, world)
    ms_s1 = timed_loop(s1.step, args.steps, 2, world) if s1 is not None else None

    # informational: the two stages of a step are independent of each other (different inputs), so a trainer may
    # run them on two streams; the memory-bound patch kernels then fill idle issue slots of the photometric kernels.
    # NOT the headline: `value` is the plain sequential step above.
    ms_overlap = None
    if s1 is not None:
        side = torch.cuda.Stream(device=device)

        def step_overlapped():
            fork = torch.cuda.Event()
            fork.record()
            side.wait_event(fork)
            with torch.cuda.stream(side):
                s1.step()
                join = torch.cuda.Event()
                join.record(side)
            out = s2.step()
            torch.cuda.current_stream().wait_event(join)
            return out

        ms_overlap = timed_loop(step_overlapped, args.steps, 2, world)

    # dominant kernel, timed live with CUDA events around its launches on the launching stream: the one-launch
    # multi-scale objective kernel (photo_ms_kernel, csrc/photo_ms.cu) -- or, with DMH_MULTISCALE=0, the per-scale
    # kernel (one launch per scale, alternating two streams: span of the step's group / launches in it)
    from depthmodelhardening_b200 import ops
    ops.KERNEL_EVENTS = []
    for _ in range(8):
        s2.step()
    torch.cuda.synchronize()
    ev_ms = [(a, b) for (name, a, b) in ops.KERNEL_EVENTS if name == "photo_ms"]
    ev = [(a, b) for (name, a, b) in ops.KERNEL_EVENTS if name == "photo_scale"]
    ops.KERNEL_EVENTS = None
    S_ = len(SCALES)
    F = len(FRAME_IDS) - 1
    sigma_disp = sum(4.0 ** (-s) for s in range(S_))
    if ev_ms:
        # (the events bracket the launch on the launching stream: a host-side pause between the first event and the
        # launch -- the queue is empty at the start of this short loop -- shows up as kernel time; the first launch is
        # dropped and the MEDIAN of the rest is reported)
        kt = sorted(a.elapsed_time(b) for (a, b) in ev_ms[1:])
        kt = [kt[len(kt) // 2]] * len(kt)
        kernel_name = "photo_ms_kernel<FASTDIV, PIPE=1, 2 CTAs/SM> (dmh_photo_multiscale: all %d scales in one launch)" % S_
        # compulsory traffic of the launch (fp32): target 12 + packed source 16 (the (B,H,W,4) layout it is handed)
        # + identity loss 4 + per scale (tie-break noise 4 + gradient 4) + the disparity pyramid 4 * sum 4^-s
        k_px = 12 + 16 + 4 + S_ * (4 + 4) + 4 * sigma_disp
    else:
        kt = []
        for i in range(0, len(ev) - S_ + 1, S_):
            grp = ev[i:i + S_]
            span = max(grp[0][0].elapsed_time(b) for (_, b) in grp) - min(grp[0][0].elapsed_time(a) for (a, _) in grp)
            kt += [span / S_] * S_
        kernel_name = "photo_fast_kernel<TMA,FASTDIV,PACKED,UP> (dmh_photo_scale, one launch per scale)"
        k_px = 12 + 12 * F + 4 + 4 * F + 4 * F + 4
    kms = sum(kt) / max(len(kt), 1)
    k_bytes = k_px * B * H * W
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = k_bytes / (kms * 1e-3) / 1e9 if kms > 0 else 0.0
    step_bytes, per_px = algorithmic_bytes(B, F, len(SCALES))
    if s1 is not None:
        step_bytes_total = step_bytes + 14.8e6 * B
    else:
        step_bytes_total = step_bytes

    # end to end: pinned host inputs -> H2D -> step -> D2H loss, EVERY step, through the public Python API.
    # Double-buffered: a copy stream uploads batch i+1 while the compute stream works on batch i (every byte is
    # still copied inside the timed region; the pipeline only overlaps the copy with the previous step).
    def measure_e2e(frame_dtype):
        from depthmodelhardening_b200 import objective
        pin = lambda t: t.pin_memory()
        if frame_dtype == torch.uint8:
            cast = lambda t: (t * 255.0).round().clamp_(0, 255).to(torch.uint8)
        else:
            cast = (lambda t: t.to(frame_dtype)) if frame_dtype != torch.float32 else (lambda t: t)
        host = {("color",) + k: pin(cast(v)) for k, v in pb_host.color.items()}
        host.update({("disp", k): pin(v) for k, v in pb_host.disp.items()})
        host[("K",)] = pin(pb_host.K)
        host[("inv_K",)] = pin(pb_host.inv_K)
        host.update({("T", k): pin(v) for k, v in pb_host.T.items()})
        if s1 is not None:
            host[("scenes",)] = pin(cast(pt_host.scenes))
        h2d = sum(v.numel() * v.element_size() for v in host.values())
        loss_host = torch.empty((), dtype=torch.float32).pin_memory()
        # the batch dictionary lives in ONE pinned arena: one cudaMemcpyAsync per step instead of ~20
        from depthmodelhardening_b200.staging import BatchArena
        arena = BatchArena(host, device, slots=2)
        for sl_ in range(2):
            for k, v in arena.host_views(sl_).items():
                v.copy_(host[k])
        slots = [arena.device_views(i) for i in range(2)]
        for sl in slots:
            for k in sl:
                if k[0] == "disp":
                    sl[k].requires_grad_(True)
        f32buf = {}
        if frame_dtype == torch.uint8:
            from depthmodelhardening_b200.staging import unpack_u8
            f32buf = {k: torch.empty(v.shape, dtype=torch.float32, device=device) for k, v in host.items()
                      if v.dtype == torch.uint8}
        copy_stream = torch.cuda.Stream(device=device)
        ready = [torch.cuda.Event() for _ in range(2)]
        done = [torch.cuda.Event() for _ in range(2)]

        def upload(slot):
            with torch.cuda.stream(copy_stream), torch.no_grad():
                copy_stream.wait_event(done[slot])          # the previous user of this slot has finished
                arena.upload(slot)
                ready[slot].record(copy_stream)

        def compute(slot):
            sl = slots[slot]
            torch.cuda.current_stream().wait_event(ready[slot])
            if frame_dtype == torch.uint8:
                # bytes -> k/255 fp32 on the device (dmh_unpack_u8: the loaders' to_tensor arithmetic, bit for bit)
                sl = dict(sl)
                for k, buf in f32buf.items():
                    sl[k] = unpack_u8(sl[k], out=buf)
            color = {k[1:]: v for k, v in sl.items() if k[0] == "color"}
            disps = {k[1]: v for k, v in sl.items() if k[0] == "disp"}
            T = {k[1]: v for k, v in sl.items() if k[0] == "T"}
            for d in disps.values():
                d.grad = None
            if s1 is not None:
                s1.g.scenes = sl[("scenes",)] if frame_dtype == torch.float32 else sl[("scenes",)].float()
                s1.step()
            losses, _ = objective.photometric_losses(color, disps, sl[("K",)], sl[("inv_K",)], T, list(FRAME_IDS),
                                                     list(SCALES), H, W, noise=None, noise_mode="device")
            losses["loss"].backward()
            loss_host.copy_(losses["loss"].detach(), non_blocking=True)
            done[slot].record()

        def run_pipeline(n):
            upload(0)
            for i in range(n):
                if i + 1 < n:
                    upload((i + 1) % 2)
                compute(i % 2)

        run_pipeline(3)                                       # warm-up
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()
        n_e2e = max(4, args.steps // 2)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        copy_stream.wait_event(e0)
        run_pipeline(n_e2e)
        e1.record()
        torch.cuda.synchronize()
        ms_e2e = e0.elapsed_time(e1) / n_e2e
        if world > 1:
            t = torch.tensor([ms_e2e], device="cuda")
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            ms_e2e = float(t.item())
        return {"value": world * B * H * W / (ms_e2e * 1e-3) / 1e6, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e, "steps": n_e2e,
               "note": "public Python API; the batch dict (frames, pyramid, disparities, K, inv_K, T, scenes) is copied "
                       "from one pinned host arena every step (staging.BatchArena, a single cudaMemcpyAsync) on a copy "
                       "stream, double-buffered against the previous step's compute; tie-break noise drawn on the device; loss read back every step"}


    # end to end from the RAW bytes (informational): the loader-side compositing (next-2) runs on the device too.
    # Host buffers per step: the 8-bit native-resolution stereo pair of every item, the 8-bit attack scenes, the
    # disparities (fp32), K / inv_K / T.  Device: unpack -> AdvBatchComposer (warp + composite + Lanczos pyramids)
    # -> stage 1 -> stage 2 (objective on the composited frames) -> loss read-back.  Same double-buffered pipeline.
    def measure_e2e_composer():
        import tempfile
        from depthmodelhardening_b200 import loader, objective, patch_ops, synth
        from depthmodelhardening_b200.staging import BatchArena, unpack_u8
        tmp = tempfile.mkdtemp(prefix="dmh_calib_")
        os.makedirs(os.path.join(tmp, "training", "calib"))
        calib = os.path.join(tmp, "training", "calib", "003086.txt")
        with open(calib, "w") as f:
            p2 = " ".join(repr(v) for v in patch_ops.KITTI_P2_003086)
            for k in ("P0", "P1", "P2", "P3"):
                f.write("%s: %s\n" % (k, p2))
            f.write("R0_rect: 1 0 0 0 1 0 0 0 1\nTr_velo_to_cam: 1 0 0 0 0 1 0 0 0 0 1 0\n")
        comp = loader.AdvBatchComposer(pt_host.obj.to(device), pt_host.mask.to(device), {"path": calib}, H, W, len(SCALES))
        comp.update_adv_obj(s1.adv.detach().clone())
        pin = lambda t: t.pin_memory()
        to_u8 = lambda t: (t * 255.0).round().clamp_(0, 255).to(torch.uint8)
        host = {("raw", 0): pin(synth.frames_u8(7000 + 10 * rank, batch=B)),
                ("raw", "s"): pin(synth.frames_u8(7001 + 10 * rank, batch=B)),
                ("scenes",): pin(to_u8(pt_host.scenes)), ("K",): pin(pb_host.K), ("inv_K",): pin(pb_host.inv_K)}
        host.update({("disp", k): pin(v) for k, v in pb_host.disp.items()})
        host.update({("T", k): pin(v) for k, v in pb_host.T.items()})
        h2d = sum(v.numel() * v.element_size() for v in host.values())
        arena = BatchArena(host, device, slots=2)
        for sl_ in range(2):
            for k, v in arena.host_views(sl_).items():
                v.copy_(host[k])
        slots = [arena.device_views(i) for i in range(2)]
        for sl in slots:
            for k in sl:
                if k[0] == "disp":
                    sl[k].requires_grad_(True)
        scenes_buf = torch.empty(pt_host.scenes.shape, dtype=torch.float32, device=device)
        sides = ["l" if i % 2 == 0 else "r" for i in range(B)]
        flips = [(i // 2) % 2 == 1 for i in range(B)]
        loss_host = torch.empty((), dtype=torch.float32).pin_memory()
        copy_stream = torch.cuda.Stream(device=device)
        ready = [torch.cuda.Event() for _ in range(2)]
        done = [torch.cuda.Event() for _ in range(2)]

        def upload(slot):
            with torch.cuda.stream(copy_stream), torch.no_grad():
                copy_stream.wait_event(done[slot])
                arena.upload(slot)
                ready[slot].record(copy_stream)

        def compute(slot):
            sl = slots[slot]
            torch.cuda.current_stream().wait_event(ready[slot])
            out = comp(sl[("raw", 0)], sl[("raw", "s")], sides, flips, pt_host.z0, pt_host.alpha)
            color = {(0, s_): out[("color", 0, s_)] for s_ in SCALES}
            color[("s", 0)] = out[("color", "s", 0)]
            disps = {k[1]: v for k, v in sl.items() if k[0] == "disp"}
            T = {k[1]: v for k, v in sl.items() if k[0] == "T"}
            for d in disps.values():
                d.grad = None
            s1.g.scenes = unpack_u8(sl[("scenes",)], out=scenes_buf)
            s1.step()
            losses, _ = objective.photometric_losses(color, disps, sl[("K",)], sl[("inv_K",)], T, list(FRAME_IDS),
                                                     list(SCALES), H, W, noise=None, noise_mode="device")
            losses["loss"].backward()
            loss_host.copy_(losses["loss"].detach(), non_blocking=True)
            done[slot].record()

        def run_pipeline(n):
            upload(0)
            for i in range(n):
                if i + 1 < n:
                    upload((i + 1) % 2)
                compute(i % 2)

        run_pipeline(3)
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()
        n_e2e = max(4, args.steps // 2)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        copy_stream.wait_event(e0)
        run_pipeline(n_e2e)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n_e2e
        if world > 1:
            t = torch.tensor([ms], device="cuda")
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            ms = float(t.item())
        assert bool(torch.isfinite(loss_host))
        return {"value": world * B * H * W / (ms * 1e-3) / 1e6, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                "d2h_bytes_per_step": 4, "ms_per_step": ms, "steps": n_e2e,
                "note": "OPTION, not the headline: the whole pipeline from raw bytes -- 8-bit native-resolution stereo "
                        "pairs and scenes + fp32 disparities cross PCIe, the training-batch compositing "
                        "(loader.AdvBatchComposer: warp, composite, Pillow-exact Lanczos pyramids) runs on the device "
                        "before stage 1 and stage 2; replaces the CPU DataLoader work of the reference"}

    e2e = e2e_bf16 = e2e_u8 = e2e_composer = None
    if not args.no_e2e:
        scenes_f32 = s1.g.scenes if s1 is not None else None
        e2e = measure_e2e(torch.float32)
        if not args.no_e2e_u8:
            e2e_u8 = measure_e2e(torch.uint8)
            e2e_u8["note"] = ("OPTION, not the headline: colour frames, pyramid and scenes travel as the 8-bit images the "
                              "reference's loaders decode (a quarter of the bytes) and become k/255 fp32 on the device "
                              "(dmh_unpack_u8, IEEE division == torchvision to_tensor bit for bit): lossless for 8-bit "
                              "sources; the synthetic frames are quantised to k/255 for this measurement")
        if not args.no_e2e_bf16:
            e2e_bf16 = measure_e2e(torch.bfloat16)
            e2e_bf16["note"] = ("OPTION, not the headline: colour frames, pyramid and scenes travel as bf16 (half the "
                                "bytes) and are up-cast on the device; results then carry the 2e-3 tolerance class")
        if s1 is not None and not args.no_e2e_u8:
            try:
                e2e_composer = measure_e2e_composer()
            except Exception as exc:                        # informational line: never take the bench down with it
                e2e_composer = {"error": "%s: %s" % (type(exc).__name__, exc)}
        if s1 is not None:
            s1.g.scenes = scenes_f32

    # DRAM traffic / instruction count of the dominant kernel per launch are NOT measured by this run: they are read
    # from the committed ncu capture of this command (profiles/r02_ncu_photo_ms.json, written by
    # profiles/summarize_ncu.py --json) when it describes the same kernel and batch; otherwise null
    ncu_traffic = ncu_warp_inst = None
    ncu_src = None
    try:
        cap = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_photo_ms.json")))
        if cap.get("batch") == B and bool(ev_ms) and cap.get("kernel", "").startswith("photo_ms"):
            ncu_traffic = cap.get("dram_bytes_per_launch")
            ncu_warp_inst = cap.get("warp_instructions_per_launch")
            ncu_src = "profiles/r02_ncu_photo_ms.json (%s)" % cap.get("source", "ncu --set full")
    except Exception:
        pass
    sm_clock_hz = float((clocks or {}).get("sm_mhz") or 1965.0) * 1e6
    roofline = {"bound": "hbm", "kernel": kernel_name,
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if peak else None,
                "traffic": ncu_traffic, "traffic_source": ncu_src,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6.65 TB/s",
                "kernel_ms": kms, "kernel_launches_timed": len(kt), "algorithmic_bytes_per_launch": k_bytes,
                "algorithmic_bytes_per_px": k_px,
                # continuity with round 1, whose accounting charged every scale its own copy of the target / source /
                # identity loss (40 B per pixel and scale): the same kernel time against S x 40 B/px
                "frac_round1_accounting": (40.0 * S_ * B * H * W / (kms * 1e-3) / 1e9 / peak) if (kms > 0 and ev_ms) else None,
                "step_algorithmic_bytes": step_bytes_total,
                "step_hbm_frac": step_bytes_total / (ms_step * 1e-3) / 1e9 / peak,
                "note": "DRAM traffic ~ algorithmic bytes (no re-reads) but the kernel is fp32 instruction-issue "
                        "bound, not HBM bound (see issue_frac): fusing the scales REMOVED compulsory bytes (target, "
                        "source and identity loss are read once instead of once per scale), so `frac` of the fused "
                        "launch is lower than round 1's per-scale figure although the launch is faster; "
                        "step_hbm_frac (SURVEY.md 8(d) whole-step bytes / step time) is the comparable number"}
    if ncu_warp_inst and kms > 0:
        # fraction of the SM issue slots (148 SMs x 4 schedulers x 1 warp-instruction / clock) the kernel uses
        roofline["issue_frac"] = ncu_warp_inst / (kms * 1e-3) / (148 * 4 * sm_clock_hz)
        roofline["warp_instructions_per_launch"] = ncu_warp_inst

    line = {
        "metric": METRIC, "value": world * B * H * W / (ms_step * 1e-3) / 1e6, "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[1]: monodepth2 1024x320 stereo [0,'s'], 4 scales, automask, SSIM+L1, "
                               "smoothness; step = patch PGD step (stage 1, %s update) + photometric loss fwd/bwd (stage 2)" % args.attack
                               if s1 is not None else
                               "configs[1] stage 2 only: photometric loss fwd/bwd (stage 1 not built yet)",
                   "per_gpu_batch": B, "global_batch": B * world, "height": H, "width": W, "frame_ids": list(FRAME_IDS),
                   "scales": list(SCALES), "l2_policy": "inputs (2x126 MB frames + 168 MB noise) exceed the 126 MB L2"},
        "gpu_launches": launches,
        "schedule": schedule, "ms_per_step_eager": ms_eager,
        "value_eager": world * B * H * W / (ms_eager * 1e-3) / 1e6,
        "clocks": clocks,
        "stages": {"photometric_ms": ms_s2, "patch_pgd_ms": ms_s1, "two_stream_step_ms": ms_overlap,
                   "pgd_steps_per_s": (1e3 / ms_s1) if ms_s1 else None,
                   "photometric_mpix_per_s": world * B * H * W / (ms_s2 * 1e-3) / 1e6},
        "roofline": roofline,
    }
    if e2e is not None:
        line["e2e"] = e2e
    if e2e_bf16 is not None:
        line["e2e_bf16_frames"] = e2e_bf16
    if e2e_u8 is not None:
        line["e2e_u8_frames"] = e2e_u8
    if e2e_composer is not None:
        line["e2e_composer"] = e2e_composer
    if not args.no_strong and s1 is not None:
        # north_star's scaling configuration: GLOBAL batch 32 sharded over the ranks (32/16/8/4 items per GPU)
        try:
            line["strong_scaling"] = measure_strong(args, rank, world, device, GLOBAL_BATCH)
        except Exception as exc:
            line["strong_scaling"] = {"error": "%s: %s" % (type(exc).__name__, exc)}
    if world == 1 and args.strong_shard > 1 and s1 is not None:
        try:
            em = measure_strong(args, rank, 1, device, GLOBAL_BATCH, shard=args.strong_shard)
            em["note"] = ("EMULATION on one GPU of the shard a %d-GPU strong-scaling run gives each rank (%d items), "
                          "without the collective; the N-GPU numbers are the strong_scaling records of the N-GPU runs"
                          % (args.strong_shard, GLOBAL_BATCH // args.strong_shard))
            em["value"] = em["value_eager"] = em["value_two_stream"] = None
            line["strong_shard_emulation"] = em
        except Exception as exc:
            line["strong_shard_emulation"] = {"error": "%s: %s" % (type(exc).__name__, exc)}
    if world == 1 and not args.no_strong and s1 is not None:
        try:
            line["multisource"] = measure_multisource(args, device, B)
        except Exception as exc:                            # informational: never take the bench down with it
            line["multisource"] = {"error": "%s: %s" % (type(exc).__name__, exc)}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = run_cpu_baseline(args.cpu_sample_batch or 8, s1 is not None, attack=args.attack)
    if rank == 0 and world == 1 and not args.no_gpu_eager and reference_available():
        try:
            # free this arm's buffers first: the eager reference keeps ~10 full-size tensors per scale alive
            del s2, s1
            torch.cuda.empty_cache()
            ge = gpu_eager_baseline(B, with_patch, args.attack, device)
            ge["graft_speedup"] = ge["ms_per_step"] / ms_step
            line["gpu_eager_baseline"] = ge
        except Exception as exc:                            # informational: never take the bench down with it
            line["gpu_eager_baseline"] = {"error": "%s: %s" % (type(exc).__name__, exc)}
    if world > 1:
        torch.distributed.destroy_process_group()
    sys.stdout.flush()
    if rank == 0:
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    os.close(json_fd)


if __name__ == "__main__":
    main()
