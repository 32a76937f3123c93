"""bench.py --dump-outputs.  CPU: float32 .npy files; an array larger than the per-array cap becomes the same seeded
sample of its elements in every run.  GPU: the files hold what the last timed step computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench
from tests.util import assert_close


def test_dump_outputs_writes_small_arrays_whole_and_samples_large_ones(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_MAX_ELEMENTS", 1000)
    big = torch.arange(5000, dtype=torch.float32).view(5, 1000)
    small = torch.rand(2, 3, 4, dtype=torch.float64)
    for d in ("a", "b"):
        bench.dump_outputs({"loss": torch.tensor(0.25), "small": small, "big": big}, str(tmp_path / d))
    assert sorted(os.listdir(tmp_path / "a")) == ["big.npy", "loss.npy", "small.npy"]
    s, loss = np.load(tmp_path / "a" / "small.npy"), np.load(tmp_path / "a" / "loss.npy")
    assert s.dtype == np.float32 and s.shape == (2, 3, 4) and np.array_equal(s, small.float().numpy())
    assert loss.shape == () and float(loss) == 0.25
    a, b = np.load(tmp_path / "a" / "big.npy"), np.load(tmp_path / "b" / "big.npy")
    assert a.dtype == np.float32 and a.ndim == 1 and 800 < a.size <= 1000 and np.array_equal(a, b)
    # the sample holds distinct elements in index order (big's value is its flat index)
    assert np.all(np.diff(a) > 0) and a[0] >= 0 and a[-1] < 5000


@pytest.mark.gpu
def test_dump_holds_the_outputs_of_the_captured_step(tmp_path):
    """bench.py --steps 1 --dump-outputs: the headline ran as a CUDA-graph replay (a loss kept with its autograd graph
    breaks the capture), its objective outputs equal one eager step on the same seeded inputs, and the patch step's
    scenes, mask and gradient equal one fused apply of the dumped patch."""
    from depthmodelhardening_b200 import patch_ops
    B = 2
    r = subprocess.run([sys.executable, os.path.join(bench.ROOT, "bench.py"), "--steps", "1", "--warmup", "0",
                        "--batch", str(B), "--no-e2e", "--no-strong", "--no-cpu-baseline", "--no-gpu-eager",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["schedule"].startswith("CUDA-graph replay"), line["schedule"]
    dev = torch.device("cuda:0")
    pb, pt = bench.make_host_workload(B, 0, True)
    s2 = bench.Stage2(pb, dev)
    s2.step()
    expected = s2.outputs
    assert sorted(expected) == ["grad_disp_0", "grad_disp_1", "grad_disp_2", "grad_disp_3", "loss", "loss_0", "loss_1",
                                "loss_2", "loss_3"]
    for name, t in expected.items():
        assert_close(np.load(tmp_path / (name + ".npy")), t, 1e-6, name)
    s1 = bench.Stage1(pt, dev, 1)
    patch = torch.from_numpy(np.load(tmp_path / "patch.npy")).to(dev)
    adv, mask, grad = patch_ops.apply_patch_fwd_bwd(patch, s1.g.mask, s1.g.scenes, s1.coeffs, s1.g.upstream)
    assert_close(np.load(tmp_path / "adv_scene.npy"), adv, 1e-6, "adv_scene")
    assert_close(np.load(tmp_path / "mask.npy"), mask, 1e-6, "mask")
    assert_close(np.load(tmp_path / "grad_patch.npy"), grad, 1e-5, "grad_patch")
    for name in ("pattern_pos", "pattern_neg"):
        p = np.load(tmp_path / (name + ".npy"))
        assert p.shape == tuple(patch.shape) and np.isfinite(p).all()
