#!/usr/bin/env python
"""Same-box A/B of environment settings: prints one JSON line with the stage-2 time (CUDA events), the whole step as a
two-stream CUDA-graph replay at per-GPU batch 32 (the bench headline) and at batch 4 (the shard of an 8-GPU
strong-scaling run, no collective).  The settings are environment variables read by the library / bench.py
(DMH_MULTISCALE, DMH_MULTISOURCE, DMH_S1_PRIORITY): run once per setting, e.g.
    for p in 0 1; do DMH_MULTISCALE=$p python profiles/ab.py; done"""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402


def main():
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    from depthmodelhardening_b200 import _lib
    lib = _lib.load()
    out = {"env": {k: v for k, v in os.environ.items() if k.startswith("DMH_")}}
    for B in (32, 4):
        pb, pt = bench.make_host_workload(B, 0, True)
        s2 = bench.Stage2(pb, dev)
        s1 = bench.Stage1(pt, dev, 1, "l0")
        ms2 = bench.timed_loop(s2.step, 30, 5, 1)
        graph, n = bench.capture_step(s1, s2, dev, lib, two_stream=True)
        msg = bench.timed_loop(graph.replay, 50, 10, 1)
        msg = min(msg, bench.timed_loop(graph.replay, 50, 5, 1))
        out["B%d" % B] = {"stage2_eager_ms": round(ms2, 4), "step_graph_two_stream_ms": round(msg, 4), "launches": n}
        del graph, s1, s2
        torch.cuda.empty_cache()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
