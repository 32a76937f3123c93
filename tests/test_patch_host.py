"""CPU: host-side logic of stage 1 -- corner projection (int32 truncation), the
batched fp64 homography solve against torchvision's per-item solve, start
corners, calib parsing, and the attack classes' argument / error behaviour."""
import numpy as np
import pytest
import torch

from depthmodelhardening_b200 import patch_ops, physical
from oracle.refload import CALIB_P2, write_calib
from tests.util import load_golden

P34 = np.array(CALIB_P2, dtype=np.float64).reshape(3, 4)


def test_corners_match_reference_golden():
    g = load_golden("patch")
    K = np.array([[0.58 * 1242, 0, 0.5 * 1242, 0], [0, 1.92 * 375, 0.5 * 375, 0], [0, 0, 1, 0], [0, 0, 0, 1]],
                 dtype=np.float32)
    for i, (z, a) in enumerate(zip(g["z0"].tolist(), g["alpha"].tolist())):
        assert np.array_equal(patch_ops.project_corners(z, a, P34), g["corners"][i])
        assert np.array_equal(patch_ops.project_corners(z, a, P34, K=K), g["corners_k"][i])


def test_batched_homography_solve_equals_torchvision():
    from torchvision.transforms.functional import _get_perspective_coeffs
    start = patch_ops.start_corners((260, 300))
    assert start == [[471, 57], [771, 57], [771, 317], [471, 317]]
    zs = [5.0 + 0.2 * i for i in range(25)]
    als = [-30.0 + 5.0 * (i % 13) for i in range(25)]
    ends = np.stack([patch_ops.project_corners(z, a, P34) for z, a in zip(zs, als)])
    co = patch_ops.solve_homographies(start, ends)
    assert co.shape == (25, 8) and co.dtype == torch.float32
    for i in range(25):
        ref = torch.tensor(_get_perspective_coeffs(start, ends[i].tolist()), dtype=torch.float32)
        # same fp64 gels solve; after the cast to fp32 at most 1 ulp apart
        assert torch.allclose(co[i], ref, rtol=2e-7, atol=1e-12), (i, co[i], ref)


def test_calib_reader(tmp_path):
    path = write_calib(str(tmp_path))
    P = physical.read_calib_P2(path)
    assert P.shape == (3, 4) and abs(P[0, 0] - 721.5377) < 1e-9


def test_physical_trans_asserts_canvas_size(tmp_path):
    path = write_calib(str(tmp_path))
    obj = torch.rand(1, 3, 26, 30)
    with pytest.raises(AssertionError):
        physical.PhysicalTrans(obj, torch.ones(1, 1, 26, 30), {"path": path}, (1, 3, 100, 200))
    pt = physical.PhysicalTrans(obj, torch.ones(1, 1, 26, 30), {"path": path}, (1, 3, 375, 1242))
    assert pt.pos_obj_img_start[0] == [606, 174]
    assert pt.dist_range == [5, 7, 9] and len(pt.angle_range) == 13
    with pytest.raises(ValueError):       # random.sample without replacement (physicalTrans.py:150)
        pt.project(batch_size=14)


def test_install_rebinds_reference_symbols():
    from oracle import refload
    if not refload.available():
        pytest.skip("reference tree not present")
    ref = refload.load()
    import depthmodelhardening_b200.install as dmh
    from depthmodelhardening_b200 import layers as L
    done = dmh.install(mode="fused", dataset_root=ref.calib_root)
    try:
        assert ref.layers.SSIM is L.SSIM and ref.trainer.SSIM is L.SSIM
        assert ref.trainer.Trainer.compute_losses.__name__ == "fused_compute_losses"
        assert ref.atk_l0.Phy_obj_atk_l0.__module__.startswith("depthmodelhardening_b200")
        # CPU tensors keep the reference PhysicalTrans (DataLoader workers)
        pt = ref.physicalTrans.PhysicalTrans(torch.rand(1, 3, 26, 30), torch.ones(1, 1, 26, 30),
                                             {"path": ref.calib_path}, (1, 3, 375, 1242))
        assert type(pt).__module__ == "physicalTrans"
        assert done["layers.SSIM"]
    finally:
        dmh.uninstall()
        import importlib
        importlib.reload(ref.atk_l0)
        importlib.reload(ref.atk_linf)
    assert ref.layers.SSIM is not L.SSIM


def test_placement_bbox_is_conservative():
    """Every canvas pixel that samples the patch (per the oracle's perspective warp of an all-ones
    image) lies inside the host-computed bounding box the fused apply kernels use as a skip hint: a few near
    placements, and every distance and angle the attack classes draw (range(5, 31, 2) and the non-integer distances of
    np.linspace(5, 30, 7), the 5-degree angle grid and the odd angles of range(-30, 31, 2))."""
    from oracle import patch as OQ
    zs = [5.0, 5.4, 7.0, 9.8, 6.2, 9.0]
    als = [-30.0, 30.0, 0.0, 25.0, -15.0, 5.0]
    for z in sorted(set(float(z) for z in range(5, 31, 2)) | set(np.linspace(5, 30, 7).tolist())):
        for a in range(-30, 31):
            if a % 5 == 0 or a % 2 == 0:
                zs.append(z)
                als.append(float(a))
    ones = torch.ones(1, 1, 260, 300)
    place = patch_ops.homographies(zs, als, P34)
    assert place.bbox.dtype == torch.int32 and place.bbox.shape == (len(zs), 4)
    assert place.shape == (len(zs), 8)
    padded, start = OQ.pad_to_canvas(ones)
    for i, (z, a) in enumerate(zip(zs, als)):
        end = OQ.corners_on_image(z, a, P34)
        warped = OQ.perspective_warp(padded, OQ.perspective_coeffs(start, end.tolist()))[0, 0]
        ys, xs = torch.nonzero(warped > 0, as_tuple=True)
        x0, y0, x1, y1 = place.bbox[i].tolist()
        where = "z0=%g alpha=%g" % (z, a)
        assert xs.numel() > 1000, where
        assert int(xs.min()) >= x0 and int(xs.max()) <= x1 and int(ys.min()) >= y0 and int(ys.max()) <= y1, where
        # ... and is not vacuous: within a few pixels of the true extent
        assert int(xs.min()) - x0 <= 8 and x1 - int(xs.max()) <= 8, where
        assert place.bbox_wh[0] >= x1 - x0 + 1 and place.bbox_wh[1] >= y1 - y0 + 1, where


def test_install_rebinds_every_patch_attack_class():
    """next-4: every `Phy_obj_atk*` class of the reference (nine modules) is rebound to its drop-in by install() and
    restored by uninstall()."""
    import importlib
    import os
    from oracle import refload
    if not refload.available():
        pytest.skip("reference tree not present")
    ref = refload.load()
    import depthmodelhardening_b200.install as dmh
    names = {"phy_obj_atk": "Phy_obj_atk", "phy_obj_atk_l0": "Phy_obj_atk_l0", "phy_obj_atk_l2": "Phy_obj_atk_l2",
             "phy_obj_atk_vanila": "Phy_obj_atk_vanila", "phy_obj_atk_apgd": "Phy_obj_atk_APGD",
             "phy_obj_atk_guassian": "Phy_obj_atk_guassian", "phy_obj_atk_arbi": "Phy_obj_atk_arbi",
             "phy_obj_atk_square": "Phy_obj_atk_Square", "phy_obj_atk_light": "Phy_obj_atk_light"}
    old = os.getcwd()
    os.chdir(refload.M2_DIR)
    try:
        mods = {m: importlib.import_module("torchattacks.attacks." + m) for m in names}
    finally:
        os.chdir(old)
    originals = {m: getattr(mods[m], c) for m, c in names.items()}
    for m, c in names.items():
        assert originals[m].__module__ == "torchattacks.attacks." + m, (m, originals[m].__module__)
    done = dmh.install(mode="ops", dataset_root=ref.calib_root)
    try:
        for m, c in names.items():
            assert done.get("torchattacks.attacks.%s.%s" % (m, c)), (m, sorted(done))
            assert getattr(mods[m], c).__module__ == "depthmodelhardening_b200.attacks", m
    finally:
        dmh.uninstall()
    for m, c in names.items():
        assert getattr(mods[m], c) is originals[m], m


# ---- stage 1: the span table of the patch kernels (csrc/patch.cu aa_table_kernel / aa_span3) against the per-pixel
# weight function the backward used before (aa_weight_of), restated op by op in IEEE float32
f32 = np.float32


def _aa_filter(x):
    x = abs(x)
    return f32(1.0) - x if x < f32(1.0) else f32(0.0)


def _span3(i, in_size, scale):
    """aa_span3: (lo, w0, w1, w2) of output index i."""
    support = scale if scale >= f32(1.0) else f32(1.0)
    invscale = f32(1.0) / scale if scale >= f32(1.0) else f32(1.0)
    center = f32(scale * f32(f32(i) + f32(0.5)))
    lo = max(int(f32(f32(center - support) + f32(0.5))), 0)
    n = min(min(int(f32(f32(center + support) + f32(0.5))), in_size) - lo, 3)
    w, total = [], f32(0.0)
    for j in range(3):
        wj = _aa_filter(f32(f32(f32(f32(j) + f32(f32(lo) - center)) + f32(0.5)) * invscale)) if j < n else f32(0.0)
        w.append(wj)
        total = f32(total + wj)
    if total != 0:
        w = [f32(x / total) for x in w]
    return lo, w


def _weight_of(o, in_size, scale, ci, maxt=8):
    """aa_weight_of: weight with which output index o reads input index ci."""
    support = scale if scale >= f32(1.0) else f32(1.0)
    invscale = f32(1.0) / scale if scale >= f32(1.0) else f32(1.0)
    center = f32(scale * f32(f32(o) + f32(0.5)))
    lo = max(int(f32(f32(center - support) + f32(0.5))), 0)
    n = min(min(int(f32(f32(center + support) + f32(0.5))), in_size) - lo, maxt)
    if ci < lo or ci >= lo + n:
        return f32(0.0)
    total, mine = f32(0.0), f32(0.0)
    for j in range(n):
        w = _aa_filter(f32(f32(f32(f32(j) + f32(f32(lo) - center)) + f32(0.5)) * invscale))
        total = f32(total + w)
        if lo + j == ci:
            mine = w
    return f32(mine / total) if total != 0 else mine


@pytest.mark.parametrize("in_size,out_size", [(1242, 1024), (375, 320), (100, 81), (64, 64), (97, 70)])
def test_span_table_equals_the_per_pixel_weight_function(in_size, out_size):
    """Every (output index, input index) pair: the table entry the patch kernels read == aa_weight_of, bit for bit, for
    scale factors below 1.5 (3-tap spans); the weights of a span sum to 1 within rounding."""
    scale = f32(f32(in_size) / f32(out_size))
    assert scale < 1.5
    for o in range(out_size):
        lo, w = _span3(o, in_size, scale)
        assert abs(float(sum(w, f32(0.0))) - 1.0) < 1e-6
        for ci in range(max(lo - 2, 0), min(lo + 5, in_size)):
            d = ci - lo
            tab = w[d] if 0 <= d < 3 else f32(0.0)
            ref = _weight_of(o, in_size, scale, ci)
            assert tab.tobytes() == ref.tobytes(), (o, ci, float(tab), float(ref))
