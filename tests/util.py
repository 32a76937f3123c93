"""Shared comparison helpers for the parity tests."""
import os

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# Measured parity numbers, one record per comparison: tests/conftest.py tags them with the running test and writes
# them to $DMH_PARITY_REPORT at the end of the session (committed per round as profiles/rNN_parity_errors.json, so
# that a regression INSIDE the tolerance is visible).
REPORT = []
CURRENT_TEST = [""]


def _record(kind, what, **numbers):
    REPORT.append(dict(test=CURRENT_TEST[0], kind=kind, what=what, **{k: float(v) for k, v in numbers.items()}))


def load_golden(name):
    return dict(np.load(os.path.join(GOLDEN, name + ".npz")))


def to_np(x):
    if torch.is_tensor(x):
        return x.detach().cpu().double().numpy()
    return np.asarray(x, dtype=np.float64)


def rel_err(a, b):
    """max |a-b| relative to max |b| (the tolerance BASELINE.json states is
    'relative'; images/losses/gradients are compared on their own scale)."""
    a, b = to_np(a), to_np(b)
    assert a.shape == b.shape, (a.shape, b.shape)
    scale = max(float(np.max(np.abs(b))), 1e-30)
    return float(np.max(np.abs(a - b))) / scale


def mismatch_fraction(a, b, rtol):
    a, b = to_np(a), to_np(b)
    scale = max(float(np.max(np.abs(b))), 1e-30)
    return float(np.mean(np.abs(a - b) > rtol * scale))


def assert_close(a, b, rtol, what="", max_outlier_frac=0.0, outlier_rtol=None):
    """All elements within rtol*max|b|, except at most `max_outlier_frac` of them
    (coordinate-floor discontinuities, SURVEY.md section 7), which must still be
    within `outlier_rtol`."""
    e = rel_err(a, b)
    _record("close", what, rel_err=e, rtol=rtol, beyond_rtol_frac=mismatch_fraction(a, b, rtol) if e > rtol else 0.0)
    if e <= rtol:
        return e
    if max_outlier_frac > 0.0:
        frac = mismatch_fraction(a, b, rtol)
        assert frac <= max_outlier_frac, "%s: %.3g of elements beyond rtol=%g (max rel err %.3g)" % (what, frac, rtol, e)
        if outlier_rtol is not None:
            assert e <= outlier_rtol, "%s: outlier rel err %.3g > %g" % (what, e, outlier_rtol)
        return e
    raise AssertionError("%s: rel err %.3g > %g" % (what, e, rtol))


def assert_close_arb(a, ref32, ref64, rtol, what=""):
    """Arbitrated comparison (SURVEY.md 7/8(c): fp64 re-run of the same code as
    arbiter).  Pass if within rtol of the fp32 oracle; otherwise the CUDA result
    must be within rtol of the fp64 truth, or at least as close to it as the fp32
    oracle itself is (+20 %) -- i.e. the disagreement is fp32 rounding of the
    reference, not an error of the kernel."""
    e32 = rel_err(a, ref32)
    if e32 <= rtol:
        _record("close_arb", what, rel_err_vs_fp32=e32, rtol=rtol)
        return e32
    e64 = rel_err(a, ref64)
    eref = rel_err(ref32, ref64)
    _record("close_arb", what, rel_err_vs_fp32=e32, rel_err_vs_fp64=e64, oracle32_vs_fp64=eref, rtol=rtol)
    assert e64 <= max(rtol, 1.2 * eref), "%s: rel err vs fp32 oracle %.3g, vs fp64 %.3g (oracle32 vs fp64 %.3g)" % (
        what, e32, e64, eref)
    return e32


def assert_grad_close(a, ref32, ref64, rtol, what="", outlier_frac=2e-3, slack=2.0):
    """Gradient comparison arbitrated by the fp64 oracle.

    The fp32 reference's own gradients differ from the fp64 run of the same code
    by 2-5e-5 relative (measured: tests/golden README) -- more than the 1e-5
    target -- so an fp32 kernel with a different (fused) op order cannot be
    closer than that to the fp32 reference.  Criterion: accept if within rtol of
    the fp32 oracle; otherwise, allowing `outlier_frac` of the elements to be
    coordinate-floor ties (SURVEY.md section 7), every other element must be
    within max(rtol, slack * reference-noise) of the fp64 truth, where
    reference-noise is the fp32 oracle's own (1 - outlier_frac)-quantile error
    against fp64."""
    e32 = rel_err(a, ref32)
    if e32 <= rtol:
        _record("grad", what, rel_err_vs_fp32=e32, rtol=rtol, elements=float(np.asarray(to_np(ref32)).size))
        return e32
    a_, r32, r64 = to_np(a), to_np(ref32), to_np(ref64)
    scale = max(float(np.max(np.abs(r64))), 1e-30)
    ea = np.abs(a_ - r64).ravel() / scale
    er = np.abs(r32 - r64).ravel() / scale
    noise = float(np.quantile(er, 1.0 - outlier_frac)) if er.size > 1 else float(er.max())
    thr = max(rtol, slack * noise)
    bad = int(np.sum(ea > thr))
    # knife-edge pixels (coordinate floor(), automask near-ties): a fraction, but never fewer than 2 elements
    # (small tensors) unless outliers are disabled
    allowed = 0 if outlier_frac == 0.0 else max(2, int(np.ceil(outlier_frac * er.size)))
    _record("grad", what, rel_err_vs_fp32=e32, rel_err_vs_fp64_max=float(ea.max()),
            rel_err_vs_fp64_p999=float(np.quantile(ea, 0.999)), oracle32_noise=noise, threshold=thr,
            outliers=bad, outliers_allowed=allowed, elements=er.size, rtol=rtol)
    assert bad <= allowed, "%s: %d of %d elements beyond %.3g of fp64 (allowed %d; vs fp32 oracle %.3g; oracle noise %.3g)" % (
        what, bad, er.size, thr, allowed, e32, noise)
    return e32


def assert_selection_close(sel, ref, what="argmin", frac=1e-4):
    """Automask / argmin selections: exact up to float near-ties (|a-b| ~ 1e-7 decided by the 1e-5 noise)."""
    sel, ref = np.asarray(sel), np.asarray(ref)
    bad = int(np.sum(sel != ref))
    allowed = max(2, int(np.ceil(frac * sel.size)))
    _record("selection", what, differ=bad, allowed=allowed, elements=sel.size)
    assert bad <= allowed, "%s: %d of %d selections differ (allowed %d)" % (what, bad, sel.size, allowed)


def assert_within(got, ref, bound, what, mask=None):
    """|got - ref| <= bound for every element (float64 arithmetic); `mask` selects the elements compared."""
    got, ref, bound = got.detach().double(), ref.detach(), bound.detach()
    assert torch.isfinite(got).all(), "%s: non-finite elements" % what
    err = (got - ref).abs()
    bad = err > bound
    if mask is not None:
        bad &= mask
    n = int(bad.sum())
    ratio = err / bound.clamp_min(1e-300)
    compared = ratio if mask is None else ratio[mask]
    _record("within", what, worst_over_bound=float(compared.max()) if compared.numel() else 0.0, outside=n,
            elements=compared.numel())
    if n:
        idx = tuple(int(i) for i in bad.nonzero()[0])
        ratio = float(ratio[bad].max())
        raise AssertionError("%s: %d of %d elements beyond the rounding bound (worst %.3g x the bound; first at %s: "
                             "got %r, expected %r, bound %.3g)" % (what, n, bad.numel(), ratio, idx, float(got[idx]),
                                                                   float(ref[idx]), float(bound[idx])))


def up_weights(n_out, n_in):
    """(n_out, n_in) float64 matrix of F.interpolate(bilinear, align_corners=False) weights with the kernels' fp32
    arithmetic (dmh_common.cuh up_tap, compiled to src = fma(in/out, dst + 0.5, -0.5): one rounding), l1 = src - i0,
    l0 = 1 - l1, and a tap clamped at the last pixel counts l0 + l1 (added in fp32)."""
    sc = np.float32(n_in) / np.float32(n_out)
    t = np.arange(n_out, dtype=np.float32) + np.float32(0.5)
    src = (np.float64(sc) * t.astype(np.float64) - 0.5).astype(np.float32)     # exact product, one rounding
    src = np.maximum(src, np.float32(0.0))
    i0 = np.minimum(src.astype(np.int64), n_in - 1)
    i1 = np.where(i0 < n_in - 1, i0 + 1, i0)
    l1 = (src - i0.astype(np.float32)).astype(np.float32)
    l0 = (np.float32(1.0) - l1).astype(np.float32)
    A = np.zeros((n_out, n_in))
    r = np.arange(n_out)
    same = i0 == i1
    A[r, i0] = np.where(same, (l0 + l1).astype(np.float32), l0)
    A[r[~same], i1[~same]] = l1[~same]
    return A
