"""Training-batch compositing (SURVEY.md 8(f) next-2): `MonoDataset.prep_adv_data` + `preprocess`
(DepthNetworks/monodepth2/datasets/mono_dataset.py:186-265, 119-144) on the device.

Byte / integer work is compared BIT-EXACTLY: the Lanczos resize against the oracle restatement of Pillow's
fixed-point resampling (itself pinned to the installed Pillow, the third-party owner of that arithmetic) and the
composite + 8-bit quantisation on identical fp32 inputs.  End to end the only floating-point step is the
perspective warp of the patch (<= 1e-5 relative between the CUDA kernel and torch's CPU grid_sample, tested in
test_gpu_patch.py); a difference there can move a composited pixel across a truncation boundary, so the full
pipeline is held to: identical outside the patch, <= 1 grey level on < 1 % of the bytes.
"""
import zlib

import numpy as np
import pytest
import torch

from depthmodelhardening_b200 import synth
from oracle import loader_compose as LC
from oracle import pil_resize as R
from oracle.refload import CALIB_P2, write_calib
from tests.util import load_golden

P34 = np.array(CALIB_P2, dtype=np.float64).reshape(3, 4)
H, W, S = 320, 1024, 4
# (side, do_flip, z0, alpha) -- the cases of oracle/make_golden_loader.py
CASES = [("l", False, 7, -10), ("r", False, 5, 15), ("l", True, 9, 0), ("r", True, 7, 25)]
SIZES = [(375, 1242, 320, 1024), (320, 1024, 160, 512), (160, 512, 80, 256), (80, 256, 40, 128),
         (375, 1242, 192, 640), (100, 333, 37, 53), (64, 64, 64, 32), (50, 70, 25, 70), (33, 47, 90, 121),
         (7, 5, 3, 2), (50, 70, 50, 70), (375, 1242, 190, 640), (120, 64, 40, 32), (97, 130, 45, 100)]


def crc(a):
    return np.uint32(zlib.crc32(np.ascontiguousarray(a).tobytes()))


def as_u8(t):
    """fp32 k/255 tensor -> the bytes it came from (exact: to_tensor output)."""
    u8 = (t.detach().cpu() * 255.0).round().to(torch.uint8)
    assert torch.equal(u8.float().div(255), t.detach().cpu()), "not a to_tensor image (k/255)"
    return u8.numpy()


def patches():
    pbt = synth.patch_batch(batch=1, seed=0)
    return pbt.obj, synth.rand(pbt.obj.shape, 78), pbt.mask


# ----------------------------------------------------------------------------- CPU: oracle pins, host logic
@pytest.mark.parametrize("size", SIZES)
def test_oracle_resize_equals_pillow(size):
    """The oracle's restatement of Resample.c == the installed Pillow, bit for bit (random + saturated structure)."""
    from PIL import Image
    ih, iw, oh, ow = size
    rng = np.random.default_rng(ih * 1000 + ow)
    imgs = [rng.integers(0, 256, (3, ih, iw), dtype=np.uint8), np.zeros((3, ih, iw), np.uint8)]
    imgs[1][:, ::7, :] = 255
    imgs[1][:, :, ::5] = 255
    for img in imgs:
        pil = Image.fromarray(np.transpose(img, (1, 2, 0))).resize((ow, oh), Image.LANCZOS)
        assert np.array_equal(R.resize_lanczos_u8(img, oh, ow), np.transpose(np.asarray(pil), (2, 0, 1)))


@pytest.mark.parametrize("n", [(1242, 1024), (375, 320), (1024, 512), (320, 160), (333, 53), (47, 121), (5, 2)])
def test_product_coefficients_equal_oracle(n):
    """loader.lanczos_coefficients (host side of dmh_lanczos_u8) produces Pillow's integers."""
    from depthmodelhardening_b200 import loader
    b, k = loader.lanczos_coefficients(*n)
    bo, ko = R.coefficients(*n)
    assert b.dtype == np.int32 and k.dtype == np.int32
    assert np.array_equal(b, bo) and np.array_equal(k, ko)
    assert int(np.abs(k.astype(np.int64)).sum(1).max()) * 255 < 2 ** 31      # the kernels accumulate in int32


@pytest.mark.parametrize("ci", range(len(CASES)))
def test_oracle_composer_matches_reference_golden(ci):
    """oracle/loader_compose.prep_item == the unmodified MonoDataset.prep_adv_data + preprocess: CRC of every
    pyramid level of every dictionary entry (tests/golden/loader_compose.npz, oracle/make_golden_loader.py)."""
    g = load_golden("loader_compose")
    side, flip, z0, alpha = CASES[ci]
    ben, adv, mask = patches()
    c0, cs = synth.frames_u8(1000 + 2 * ci)[0].numpy(), synth.frames_u8(1001 + 2 * ci)[0].numpy()
    out = LC.prep_item(c0, cs, side, flip, z0, alpha, adv, ben, mask, P34, H, W, S)
    n = 0
    for k, v in out.items():
        name = "c%d_%s_%s_%d" % ((ci,) + k)
        if k[0] == "objdepth":
            assert np.array_equal(v.numpy(), g["c%d_objdepth" % ci])
            continue
        u8 = as_u8(v)
        assert int(u8.astype(np.int64).sum()) == int(g[name + "_sum"]), name
        assert crc(u8) == g[name + "_crc"], name
        n += 1
    assert n == 4 * S + 2


@pytest.mark.parametrize("n", [(1242, 1024), (1024, 512), (375, 320), (47, 121)])
def test_dp4a_weight_split_is_exact(n):
    """The arithmetic identity behind lanczos_h_dp4a_kernel, emulated in integer numpy: every 22-bit weight splits
    into k2 * 65536 + k1 * 256 + k0 (k0, k1 unsigned bytes, k2 a signed byte), so a span is three 8-bit dot products
    whose recombination (in wrapping 32-bit arithmetic, as the kernel does it) equals Pillow's 32-bit accumulator."""
    from depthmodelhardening_b200 import loader
    bounds, kk = loader.lanczos_coefficients(*n)
    k = kk.astype(np.int64)
    k0, k1, k2 = k & 0xff, (k >> 8) & 0xff, k >> 16                 # arithmetic shift: k2 is signed
    assert np.array_equal(k2 * 65536 + k1 * 256 + k0, k)
    assert k2.min() >= -128 and k2.max() <= 127
    rng = np.random.default_rng(n[0])
    for px in (rng.integers(0, 256, kk.shape), np.full(kk.shape, 255), np.zeros(kk.shape, np.int64)):
        px = px.astype(np.int64)
        direct = (1 << 21) + (px * k).sum(1)
        d0, d1, d2 = (px * k0).sum(1), (px * k1).sum(1), (px * k2).sum(1)
        wrapped = ((1 << 21) + d0 + (d1 << 8) + ((d2 << 16) & 0xffffffff)) & 0xffffffff
        wrapped = np.where(wrapped >= 1 << 31, wrapped - (1 << 32), wrapped)     # reinterpret as int32
        assert np.array_equal(wrapped, direct)
        assert np.abs(direct).max() < 1 << 31


@pytest.mark.parametrize("n", [(375, 320), (320, 160), (160, 80), (80, 40), (375, 190), (375, 192), (97, 45)])
def test_row_group_weight_table_covers_every_span(n):
    """Host-side restatement of lanczos_v_group_kernel's weight table: for every group of 8 output rows the union of
    the spans starts at the first row's span, fits the launcher's bound (the formula dmh_lanczos_u8 uses to choose
    the kernel) and the zero-padded table reproduces each output's own weighted sum."""
    from depthmodelhardening_b200 import loader
    G, TS = 8, 32
    in_h, out_h = n
    bounds, kk = loader.lanczos_coefficients(in_h, out_h)
    ksize = kk.shape[1]
    group_span = ((G - 1) * in_h + out_h - 1) // out_h + ksize + 1          # as in dmh_lanczos_u8
    col = np.random.default_rng(in_h).integers(0, 256, in_h).astype(np.int64)
    for yo0 in range(0, out_h, G):
        last = min(yo0 + G, out_h) - 1
        ylo, yhi = int(bounds[yo0, 0]), int(bounds[last, 0] + bounds[last, 1])
        assert all(bounds[yo0 + g, 0] >= ylo and bounds[yo0 + g, 0] + bounds[yo0 + g, 1] <= yhi
                   for g in range(last - yo0 + 1))
        assert yhi - ylo <= group_span
        if group_span > TS:
            continue                                                         # the launcher takes the per-row kernel
        table = np.zeros((TS, G), dtype=np.int64)
        for g in range(last - yo0 + 1):
            lo, cnt = bounds[yo0 + g]
            table[lo - ylo:lo - ylo + cnt, g] = kk[yo0 + g, :cnt]
        acc = (table[:yhi - ylo] * col[ylo:yhi, None]).sum(0)
        for g in range(last - yo0 + 1):
            lo, cnt = bounds[yo0 + g]
            assert acc[g] == int((kk[yo0 + g, :cnt].astype(np.int64) * col[lo:lo + cnt]).sum())


def test_oracle_enhance_equals_pillow():
    """Groundwork for the colour jitter (DESIGN.md section 9): oracle/pil_enhance.py restates the four ColorJitter
    steps on 8-bit PIL images (mono_dataset.py:297, 344-350 -> torchvision functional_pil -> PIL.ImageEnhance /
    convert('HSV')) and equals the installed Pillow / torchvision bit for bit."""
    import torchvision.transforms.functional as TF
    from PIL import Image
    from oracle import pil_enhance as E
    rng = np.random.default_rng(3)
    rand_img = rng.integers(0, 256, (3, 61, 83), dtype=np.uint8)
    rand_img[:, :4] = rand_img[0:1, :4]                                   # grey pixels (max == min)
    # a dense sweep of the colour cube: every (r, g) pair with 17 blue levels -> 1.1 M colours
    r, g, b = np.meshgrid(np.arange(256), np.arange(256), np.arange(0, 256, 15), indexing="ij")
    cube = np.stack([r.reshape(1024, -1), g.reshape(1024, -1), b.reshape(1024, -1)]).astype(np.uint8)
    for img in (rand_img, cube):
        pil = Image.fromarray(np.ascontiguousarray(np.transpose(img, (1, 2, 0))))
        as_np = lambda im: np.transpose(np.asarray(im), (2, 0, 1))
        hsv = as_np(pil.convert("HSV"))
        assert np.array_equal(E.rgb_to_hsv(img), hsv)
        back = Image.fromarray(np.ascontiguousarray(np.transpose(hsv, (1, 2, 0))), "HSV").convert("RGB")
        assert np.array_equal(E.hsv_to_rgb(hsv), as_np(back))
        for f in (0.8, 0.8731, 1.0, 1.1999, 1.2, 0.0, 0.5, 1.7):
            assert np.array_equal(E.brightness(img, f), as_np(TF.adjust_brightness(pil, f))), ("brightness", f)
            assert np.array_equal(E.contrast(img, f), as_np(TF.adjust_contrast(pil, f))), ("contrast", f)
            assert np.array_equal(E.saturation(img, f), as_np(TF.adjust_saturation(pil, f))), ("saturation", f)
        for f in (-0.1, -0.0371, 0.0, 0.05, 0.1, 0.5, -0.5):
            assert np.array_equal(E.hue(img, f), as_np(TF.adjust_hue(pil, f))), ("hue", f)


def _jitter_cases():
    """(fn_idx, b, c, s, h) tuples: every position of the contrast step, factors inside / outside [0, 1], None factors."""
    import itertools
    rng = np.random.default_rng(9)
    cases = []
    for perm in list(itertools.permutations(range(4)))[::3]:
        cases.append((list(perm), float(rng.uniform(0.8, 1.2)), float(rng.uniform(0.8, 1.2)), float(rng.uniform(0.8, 1.2)),
                      float(rng.uniform(-0.1, 0.1))))
    cases.append(([1, 0, 3, 2], 1.7, 0.3, 0.0, -0.5))
    cases.append(([3, 2, 1, 0], None, 1.1, None, 0.07))
    cases.append(([0, 1, 2, 3], 0.9, None, 1.15, None))
    return cases


def test_oracle_jitter_equals_torchvision_colorjitter():
    """oracle/pil_enhance.jitter (the composition `ColorJitter.forward` applies, in the drawn order) against
    torchvision's own functional chain on the PIL image, bit for bit -- incl. the contrast step's mean grey level
    of the PARTIALLY jittered image."""
    import torchvision.transforms.functional as TF
    from PIL import Image
    from oracle import pil_enhance as E
    rng = np.random.default_rng(4)
    img = rng.integers(0, 256, (3, 47, 65), dtype=np.uint8)
    pil0 = Image.fromarray(np.ascontiguousarray(np.transpose(img, (1, 2, 0))))
    for (fn_idx, bf, cf, sf, hf) in _jitter_cases():
        pil = pil0
        for fn_id in fn_idx:                                   # torchvision ColorJitter.forward
            if fn_id == 0 and bf is not None:
                pil = TF.adjust_brightness(pil, bf)
            elif fn_id == 1 and cf is not None:
                pil = TF.adjust_contrast(pil, cf)
            elif fn_id == 2 and sf is not None:
                pil = TF.adjust_saturation(pil, sf)
            elif fn_id == 3 and hf is not None:
                pil = TF.adjust_hue(pil, hf)
        want = np.transpose(np.asarray(pil), (2, 0, 1))
        assert np.array_equal(E.jitter(img, fn_idx, bf, cf, sf, hf), want), (fn_idx, bf, cf, sf, hf)


def test_composer_rejects_cpu_tensors():
    from depthmodelhardening_b200 import loader
    with pytest.raises(RuntimeError, match="CUDA-only"):
        loader.resize_lanczos_u8(torch.zeros(3, 8, 8, dtype=torch.uint8), 4, 4)
    with pytest.raises(RuntimeError):
        loader.compose_u8(torch.zeros(1, 3, 8, 8, dtype=torch.uint8), torch.zeros(1, 3, 8, 8), torch.zeros(1, 1, 8, 8))


# ----------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def dev():
    from depthmodelhardening_b200 import _lib
    _lib.load()
    return torch.device("cuda:0")


@pytest.mark.gpu
@pytest.mark.parametrize("size", SIZES)
def test_cuda_resize_is_bit_exact(dev, size):
    from depthmodelhardening_b200 import loader
    ih, iw, oh, ow = size
    rng = np.random.default_rng(ih + 7 * ow)
    img = rng.integers(0, 256, (2, 3, ih, iw), dtype=np.uint8)
    img[1, :, ::3, :] = 255
    img[1, :, 1::3, :] = 0
    out = loader.resize_lanczos_u8(torch.from_numpy(img).to(dev), oh, ow)
    assert out.shape == (2, 3, oh, ow) and out.dtype == torch.uint8
    assert np.array_equal(out.cpu().numpy(), R.resize_lanczos_u8(img, oh, ow))
    # to_tensor fused into the last pass (every kernel variant: row-group / 4-column / scalar vertical pass,
    # horizontal-only, no resize at all): the same bytes and exactly byte / 255
    out2, f32 = loader.resize_lanczos_u8(torch.from_numpy(img).to(dev), oh, ow, want_f32=True)
    assert torch.equal(out2, out) and f32.dtype == torch.float32
    assert torch.equal(f32.cpu(), out.cpu().to(torch.float32).div(255))


@pytest.mark.gpu
def test_cuda_pyramid_full_batch_properties(dev):
    """Full size (B=32 frames, the loader's four levels): every item equals the oracle on a sample of items,
    a constant image stays constant (weights sum to 2^22 per output) and items do not leak into each other."""
    from depthmodelhardening_b200 import loader
    B = 32
    frames = synth.frames_u8(77, batch=B)
    lv = loader.pyramid_u8(frames.to(dev), H, W, S)
    assert [tuple(l.shape) for l in lv] == [(B, 3, H >> i, W >> i) for i in range(S)]
    for b in (0, 17, 31):
        ref = R.pyramid_u8(frames[b].numpy(), H, W, S)
        for i in range(S):
            assert np.array_equal(lv[i][b].cpu().numpy(), ref[i]), (b, i)
    const = torch.full((2, 3, 375, 1242), 201, dtype=torch.uint8, device=dev)
    for l in loader.pyramid_u8(const, H, W, S):
        assert int(l.min()) == 201 and int(l.max()) == 201


@pytest.mark.gpu
@pytest.mark.parametrize("flip", [False, True])
def test_cuda_compose_is_bit_exact_on_identical_inputs(dev, flip):
    """dmh_compose_u8 against torch's CPU arithmetic on the SAME fp32 warped patch / mask (the oracle's)."""
    from depthmodelhardening_b200 import loader
    ben, adv, mask = patches()
    K = LC.adv_K()
    z0, al = [5.0, 8.5, 9.0], [-25.0, 0.0, 30.0]
    objw, maskw, _ = LC.OQ.project_patch(adv, mask, z0, al, P34, K=K, T=LC.STEREO_T)
    scenes = synth.frames_u8(31, batch=3)
    fl = [flip, not flip, flip]
    ref = np.stack([LC.compose_u8(scenes[i].numpy(), objw[i:i + 1], maskw[i:i + 1], fl[i]) for i in range(3)])
    out = loader.compose_u8(scenes.to(dev), objw.to(dev), maskw.to(dev),
                            torch.tensor([int(f) for f in fl], dtype=torch.int32))
    assert np.array_equal(out.cpu().numpy(), ref)
    m3 = maskw.expand(-1, 3, -1, -1).contiguous()
    refm = np.stack([LC.to_pil_u8(torch.flip(m3[i], [2]) if fl[i] else m3[i]) for i in range(3)])
    outm = loader.compose_u8(None, m3.to(dev), None, torch.tensor([int(f) for f in fl], dtype=torch.int32))
    assert np.array_equal(outm.cpu().numpy(), refm)


@pytest.mark.gpu
def test_cuda_fused_compose_equals_warp_then_compose(dev):
    """dmh_compose_patch_u8 (warp inside, two patches, mask image) == dmh_perspective_fwd + dmh_compose_u8, bit for
    bit, with and without the placement boxes, mixed flips, near and far (15 m, 29 m) placements."""
    from depthmodelhardening_b200 import loader, patch_ops
    ben, adv, mask = patches()
    ben, adv, mask = ben.to(dev), adv.to(dev), mask.to(dev)
    z0, al = [5.0, 6.5, 8.0, 9.0, 15.0, 29.0], [-30.0, -5.0, 10.0, 30.0, -20.0, 25.0]
    place = patch_ops.homographies(z0, al, P34, K=LC.adv_K(), T=LC.STEREO_T).to(dev)
    scenes = synth.frames_u8(55, batch=6).to(dev)
    flip = torch.tensor([0, 1, 1, 0, 1, 0], dtype=torch.int32)
    hw = (synth.ORI_H, synth.ORI_W)
    mw = patch_ops.perspective_batch(mask, place, hw)
    ref_a = loader.compose_u8(scenes, patch_ops.perspective_batch(adv, place, hw), mw, flip)
    ref_b = loader.compose_u8(scenes, patch_ops.perspective_batch(ben, place, hw), mw, flip)
    ref_m = loader.compose_u8(None, mw, None, flip)
    for pl in (place, place.coeffs):
        a, b, m = loader.compose_patch_u8(scenes, adv, ben, mask, pl, flip, want_mask=True)
        assert torch.equal(a, ref_a) and torch.equal(b, ref_b) and torch.equal(m, ref_m)
    a, b, m = loader.compose_patch_u8(scenes, adv, None, mask, place, flip)
    assert torch.equal(a, ref_a) and b is None and m is None
    # a scene buffer at an odd address takes the one-pixel-per-thread instantiation: same bytes
    odd = torch.empty(scenes.numel() + 1, dtype=torch.uint8, device=dev)[1:].view(scenes.shape)
    odd.copy_(scenes)
    assert odd.data_ptr() % 2 == 1 and odd.is_contiguous()
    a, b, m = loader.compose_patch_u8(odd, adv, ben, mask, place, flip, want_mask=True)
    assert torch.equal(a, ref_a) and torch.equal(b, ref_b) and torch.equal(m, ref_m)
    assert int((ref_a != ref_b).sum()) > 10000                 # the patches are visible
    with pytest.raises(RuntimeError, match="Batch size"):
        loader.compose_patch_u8(scenes[:3], adv, None, mask, place, None)


@pytest.mark.gpu
def test_cuda_composer_vs_oracle_and_golden(dev, tmp_path):
    """AdvBatchComposer on the four golden cases as ONE batch (mixed sides / flips / placements)."""
    from depthmodelhardening_b200 import loader
    g = load_golden("loader_compose")
    ben, adv, mask = patches()
    calib = write_calib(str(tmp_path))
    comp = loader.AdvBatchComposer(ben.to(dev), mask.to(dev), {"path": calib}, H, W, S)
    comp.update_adv_obj(adv.to(dev))
    c0 = torch.cat([synth.frames_u8(1000 + 2 * ci) for ci in range(len(CASES))])
    cs = torch.cat([synth.frames_u8(1001 + 2 * ci) for ci in range(len(CASES))])
    out = comp(c0.to(dev), cs.to(dev), [c[0] for c in CASES], [c[1] for c in CASES], [c[2] for c in CASES],
               [c[3] for c in CASES])
    assert out[("objdepth", 0, 0)].shape == (len(CASES), 1, 1)
    assert out[("color", "s", 2)] is out[("color_aug", "s", 2)]
    worst = 0.0
    for ci, (side, flip, z0, alpha) in enumerate(CASES):
        ref = LC.prep_item(c0[ci].numpy(), cs[ci].numpy(), side, flip, z0, alpha, adv, ben, mask, P34, H, W, S)
        for k, v in ref.items():
            if k[0] == "objdepth":
                assert torch.equal(out[k][ci].cpu(), v)
                continue
            got, want = as_u8(out[k][ci]).astype(np.int32), as_u8(v).astype(np.int32)
            assert got.shape == want.shape, k
            d = np.abs(got - want)
            frac = float((d > 0).mean())
            worst = max(worst, frac)
            assert d.max() <= 1 and frac < 0.01, (ci, k, int(d.max()), frac)
            # bytes that cannot see the patch are exact: everything above the horizon rows of the placement
            assert np.array_equal(got[:, : got.shape[1] // 4], want[:, : want.shape[1] // 4]), (ci, k)
            name = "c%d_%s_%s_%d" % ((ci,) + k)
            assert abs(int(got.sum()) - int(g[name + "_sum"])) <= d.size * 0.01, name
    print("composer: worst fraction of bytes off by one grey level: %.2e" % worst)
    with pytest.raises(RuntimeError, match="Batch size"):
        comp(c0.to(dev), cs.to(dev), ["l"], [False])


@pytest.mark.gpu
def test_cuda_composer_half_no_synthesis_raw_items_are_bit_exact(dev, tmp_path):
    """half_no_synthesis (mono_dataset.py:321-328): items that drew no synthesis keep their raw frames -- the whole
    device pipeline (composite with m = 0, four Lanczos levels, unpack) is then pure byte work and must equal the
    oracle bit for bit; the synthesised item of the same batch still matches its own oracle; the mask / depth
    entries are absent as in the reference (:253-255)."""
    from depthmodelhardening_b200 import loader
    ben, adv, mask = patches()
    calib = write_calib(str(tmp_path))
    comp = loader.AdvBatchComposer(ben.to(dev), mask.to(dev), {"path": calib}, H, W, S, half_no_synthesis=True)
    comp.update_adv_obj(adv.to(dev))
    c0, cs = synth.frames_u8(2000, batch=3), synth.frames_u8(2001, batch=3)
    out = comp(c0.to(dev), cs.to(dev), ["l", "r", "l"], [False, True, False], [7, 5, 9], [-10, 15, 0],
               synthesize=[False, False, True])
    assert ("color_objmask", 0, 0) not in out and ("objdepth", 0, 0) not in out
    for b in (0, 1):
        ref = LC.raw_item(c0[b].numpy(), cs[b].numpy(), H, W, S)
        assert set(ref) <= set(out)
        for k, v in ref.items():
            assert torch.equal(out[k][b].cpu(), v), (b, k)
    ref = LC.prep_item(c0[2].numpy(), cs[2].numpy(), "l", False, 9, 0, adv, ben, mask, P34, H, W, S)
    d = np.abs(as_u8(out[("color_aug", 0, 0)][2]).astype(np.int32) - as_u8(ref[("color_aug", 0, 0)]).astype(np.int32))
    assert d.max() <= 1 and float((d > 0).mean()) < 0.01
    assert int((as_u8(out[("color_aug", 0, 0)][2]) != as_u8(out[("color", 0, 0)][2])).sum()) > 1000   # patch differs



@pytest.mark.gpu
@pytest.mark.parametrize("hw", [(40, 128), (33, 37), (320, 1024)])
def test_cuda_colour_jitter_equals_oracle(dev, hw):
    """dmh_color_jitter_u8 (two launches: grey-level sums of the contrast step, then all four steps in the item's drawn
    order) against the oracle, which equals Pillow / torchvision: 8-bit output and its to_tensor image BIT-EXACT,
    every item of the batch with its own parameters, one item without augmentation."""
    from depthmodelhardening_b200 import loader
    from oracle import pil_enhance as E
    H, W = hw
    cases = _jitter_cases() + [None]
    if H * W > 100000:
        cases = cases[:3] + [None]
    B = len(cases)
    rng = np.random.default_rng(21)
    img = rng.integers(0, 256, (B, 3, H, W), dtype=np.uint8)
    img[:, :, :2] = img[:, :1, :2]                              # grey pixels
    out_u8, out_f32 = loader.color_jitter_u8(torch.from_numpy(img).to(dev), cases, want_u8=True, want_f32=True)
    torch.cuda.synchronize()
    for i, p in enumerate(cases):
        want = img[i] if p is None else E.jitter(img[i], *p)
        got = out_u8[i].cpu().numpy()
        assert np.array_equal(got, want), (i, p, int((got != want).sum()))
        assert torch.equal(out_f32[i].cpu(), torch.from_numpy(want).float() / 255.0)


@pytest.mark.gpu
def test_composer_with_colour_jitter_vs_oracle(dev):
    """AdvBatchComposer(..., color_aug=...) (mono_dataset.py:132-133, 140-144, 344-350): the "color_aug" entries and
    ("color_ben", 0, 0) are the jittered pyramid levels, the "color" entries the plain ones -- each equal to the
    oracle jitter of the composer's own 8-bit level (the levels themselves are pinned by the tests above)."""
    from depthmodelhardening_b200 import loader, synth
    from oracle import pil_enhance as E
    from oracle.refload import write_calib
    import tempfile
    calib = write_calib(tempfile.mkdtemp(prefix="dmh_calib_"))
    B = 2
    pt = synth.patch_batch(batch=B, seed=3)
    comp = loader.AdvBatchComposer(pt.obj.to(dev), pt.mask.to(dev), {"path": calib}, 320, 1024, 4)
    raw0 = synth.frames_u8(41, batch=B).to(dev)
    raws = synth.frames_u8(42, batch=B).to(dev)
    params = [([2, 0, 3, 1], 0.91, 1.13, 0.85, 0.04), None]
    kw = dict(sides=["l", "r"], do_flip=[False, True], z0_sample=[5, 7], alpha_sample=[-10, 15])
    plain = comp(raw0, raws, **kw)
    jit = comp(raw0, raws, color_aug=params, **kw)
    torch.cuda.synchronize()
    to_u8 = lambda t: (t * 255.0).round().to(torch.uint8).cpu().numpy()
    for i in range(4):
        for fid in (0, "s"):
            base = to_u8(plain[("color_aug", fid, i)])             # the un-jittered level of the same composite
            for b in range(B):
                want = base[b] if params[b] is None else E.jitter(base[b], *params[b])
                assert np.array_equal(to_u8(jit[("color_aug", fid, i)])[b], want), (i, fid, b)
            assert torch.equal(jit[("color", fid, i)], plain[("color", fid, i)])
    base = to_u8(plain[("color", 0, 0)])
    for b in range(B):
        want = base[b] if params[b] is None else E.jitter(base[b], *params[b])
        assert np.array_equal(to_u8(jit[("color_ben", 0, 0)])[b], want)
