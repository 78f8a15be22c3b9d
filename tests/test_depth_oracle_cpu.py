"""The CPU restatement of the depth-frame utilities (tests/depth_oracle.py): known answers, and the recorded reference
outputs of the calls that use no transcendental (the median fill, camera space and normals calls of
tests/test_gpu_depth_utils.py), reproduced bit for bit from the oracle alone.  The bilateral filter, whose pinned
digests need the device's exponentials, is checked there against the pins and here within a derived bound."""
from fractions import Fraction

import numpy as np
import pytest
import torch

from oracle import ref_pins
from tests import depth_oracle as O
from tests.test_gpu_depth_utils import _frames

F32 = np.float32


def _pinned():
    """The oracle behind the recorded-output check: a call whose key is not in the table, or whose outputs differ from
    the recorded ones, fails."""
    assert ref_pins.recorded()
    return ref_pins.PinnedModule(O.Module(), "depth")


def test_pins_direct_median_camspace_normals():
    """test_individual_entry_points_bit_exact's median, camera-space and normals calls."""
    m = _pinned()
    depth, intr = _frames("cpu")
    b, _, h, w = depth.shape
    filled = torch.zeros_like(depth)
    m.median_fill_depthmap(filled, depth)
    assert int((filled == 0).sum()) < int((depth == 0).sum())
    cam = torch.zeros(b, h, w, 3)
    m.convert_depth_to_cameraspace(cam, depth, intr, 0.0, 0.0)
    nrm = torch.zeros_like(cam)
    m.compute_normals(nrm, cam)                      # keyed by the camera space: found only if that was exact too
    assert int((nrm != 0).any(-1).sum()) > 0


def test_pins_median_with_unfillable_hole():
    """test_depth2normals_returns_none_when_holes_remain's median call: windows with fewer than two valid depths."""
    m = _pinned()
    depth, _ = _frames("cpu", batch=1, holes=0.0, hole_blocks=False, seed=2)
    depth[:, :, 10:70, 20:100] = 0.0
    out = torch.zeros_like(depth)
    m.median_fill_depthmap(out, depth)
    assert int((out == 0).sum()) > 0


def _two_roundings(a, b, c):
    return np.asarray(a, F32) * np.asarray(b, F32) + np.asarray(c, F32)


def _dequantise_in_double(val):
    return np.where(np.asarray(val) <= 0, 0.0, 0.001 * np.asarray(val, np.float64)).astype(F32)


@pytest.mark.parametrize("name, value", [("fma32", _two_roundings), ("dequantise", _dequantise_in_double)])
def test_pins_fail_on_a_changed_rounding(monkeypatch, name, value):
    """The anchor is sharp: one rounding changed in the oracle (the normals' FMAs as product and sum; the hole value
    0.001 * val in double) changes a pinned digest."""
    depth, intr = _frames("cpu")
    b, _, h, w = depth.shape
    m = _pinned()
    cam = torch.zeros(b, h, w, 3)
    m.convert_depth_to_cameraspace(cam, depth, intr, 0.0, 0.0)
    monkeypatch.setattr(O, name, value)
    with pytest.raises(AssertionError, match="differ from the recorded"):
        if name == "fma32":
            m.compute_normals(torch.zeros_like(cam), cam)
        else:
            m.median_fill_depthmap(torch.zeros_like(depth), depth)


# --- known answers -----------------------------------------------------------------------------------------------------

def _exact_fma32(a, b, c):
    x = Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c))
    lo = F32(float(x))                               # a neighbour of x; then pick the nearest float32, ties to even
    cands = {lo, np.nextafter(lo, F32(np.inf)), np.nextafter(lo, F32(-np.inf))}
    best = min(cands, key=lambda f: (abs(Fraction(float(f)) - x), int(np.array(f).view(np.int32)) & 1))
    return best


def test_fma32_against_fractions():
    rng = np.random.default_rng(7)
    n = 3000
    a = (rng.standard_normal(n) * np.exp2(rng.integers(-20, 20, n))).astype(F32)
    b = (rng.standard_normal(n) * np.exp2(rng.integers(-20, 20, n))).astype(F32)
    c = -(a.astype(np.float64) * b).astype(F32) * F32(1.0000001)     # heavy cancellation
    c[::3] = (rng.standard_normal(n // 3) * np.exp2(rng.integers(-40, 40, n // 3))).astype(F32)
    # products (1 + i 2^-12)(1 + j 2^-12) = 1 + (i + j) 2^-12 + ij 2^-24: exact float32 ties for odd ij, and just off a
    # tie with an addend far below the float64 ulp, where rounding the float64 sum to float32 would round twice
    i, j = np.meshgrid(np.arange(1, 16), np.arange(1, 16))
    ta = (F32(1) + i.ravel().astype(F32) * F32(2.0 ** -12)).repeat(5)
    tb = (F32(1) + j.ravel().astype(F32) * F32(2.0 ** -12)).repeat(5)
    tc = np.tile(np.array([0, 2.0 ** -60, -2.0 ** -60, 2.0 ** -40, -2.0 ** -24], F32), i.size)
    a, b, c = np.concatenate([a, ta]), np.concatenate([b, tb]), np.concatenate([c, tc])
    got = O.fma32(a, b, c)
    want = np.array([_exact_fma32(x, y, z) for x, y, z in zip(a, b, c)], F32)
    assert np.array_equal(got.view(np.int32), want.view(np.int32))
    x = F32(1 + 2.0 ** -12)                         # 1 + 2^-11 + 2^-24 + 2^-60: above the tie, so it rounds up
    assert O.fma32(x, x, F32(2.0 ** -60)) == F32(1 + 2.0 ** -11 + 2.0 ** -23)
    assert F32(float(x) * float(x) + 2.0 ** -60) == F32(1 + 2.0 ** -11)          # what float64 then float32 gives


def test_quantise_edges():
    d = np.array([1.0, 0.0015, 0.0014999999, -0.0015, -0.002, -0.0025, np.nan, 1e10, -1e10, np.inf, 2.4999999e-4,
                  0.0005, 0.00049999997], F32)
    assert O.quantise(d).tolist() == [1000, 2, 1, -1, -1, -2, 0, 2 ** 31 - 1, -2 ** 31, 2 ** 31 - 1, 0, 1, 0]
    # one rounding: 1000 x + 0.5 is just below 1, but the product rounded on its own gives exactly 1
    x = F32(0.00049999997)
    assert F32(F32(1000) * x) + F32(0.5) == F32(1.0) and O.quantise(x) == 0


@pytest.mark.parametrize("qs, want", [([], 0), ([7], 0), ([5, 9], 9), ([9, 5, 7], 9), ([4, 1, 3, 2], 3),
                                      ([6, 6, 6, 6, 6], 6), ([3, 3, 1, 1], 3), ([-1, 2], 2), ([-5, -3, -4], -3)])
def test_median_value(qs, want):
    """The ((n+1)/2)-th smallest, 0-based: the larger of two, the largest of three; 0 below two values."""
    assert O.median_value(qs) == want


def test_median_fill_window_by_hand():
    d = np.zeros((2, 3, 12), F32)
    d[0, 0, 0], d[0, 0, 2], d[0, 2, 11] = 1.25, 1.0, 2.5
    d[0, 1, 11] = -0.002                            # valid, quantises to -1
    d[0, 1, 6] = -np.inf                            # a hole, like 0
    d[1, 0, 0] = 1.25                               # frame 1: one valid depth
    out = O.median_fill(d)
    for y, x in ((0, 0), (0, 2), (2, 11), (1, 11)):
        assert out[0, y, x] == d[0, y, x]                                     # valid pixels copied
    assert out[0, 1, 0] == F32(0.001) * F32(1250)                             # window x 0-5: {1000, 1250}, the larger
    assert out[0, 1, 6] == F32(0.001) * F32(2500)                             # x 1-11: {1000, -1, 2500}, the largest
    assert out[0, 2, 8] == F32(0.001) * F32(2500)                             # x 3-13: {-1, 2500}: -1 counts
    want1 = np.zeros((3, 12), F32)
    want1[0, 0] = 1.25
    assert np.array_equal(out[1], want1)                                      # n = 1 and n = 0 windows stay holes


def test_camspace_and_normal_by_hand():
    d = np.full((1, 1, 3, 3), 2.0, F32)
    d[0, 0, 2, 1] = 3.0
    k = np.array([[100.0, 50.0, 1.0, 1.0]], F32)
    cam = O.camspace(d, k)
    assert cam[0, 0, 0].tolist() == [2.0 * F32(-0.01), 2.0 * F32(-0.02), 2.0]
    assert cam[0, 2, 1].tolist() == [0.0, 3.0 * F32(0.02), 3.0]
    # centre: a = pc - mc = (0, 0.1, 1), b = cp - cm = (0.04, 0, 0); n = a x b = (0, 0.04, -0.004), divided by -|n|
    n = O.normals(cam)[0, 1, 1].astype(np.float64)
    want = -np.array([0.0, 0.04, -0.004]) / np.hypot(0.04, 0.004)
    assert np.abs(n - want).max() < 1e-6
    assert not O.normals(cam)[0, 0].any() and not O.normals(cam)[0, :, 2].any()     # border rule
    k2 = np.concatenate([k, [[50.0, 100.0, 0.0, 2.0]]]).astype(F32)                 # intrinsics per frame
    cam2 = O.camspace(np.concatenate([d, d]), k2)
    assert np.array_equal(cam2[0], cam[0]) and cam2[1, 0, 0].tolist() == [0.0, 2.0 * F32(-0.02), 2.0]


def test_bilateral_within_bound():
    """With numpy's exponentials the oracle is within the bound that a few ulp on each Gaussian and fp32 sums allow of
    a float64 evaluation of the same filter (every tap, same skip rules)."""
    depth, _ = _frames("cpu", batch=1, h=40, w=52)
    d = depth.numpy()[0, 0].astype(np.float64)
    got = O.bilateral(depth.numpy(), 2.0, 0.1)[0, 0].astype(np.float64)
    h, w = d.shape
    r = 4
    sd, sr = float(F32(2.0)), float(F32(0.1))
    want = np.zeros_like(d)
    bound = np.zeros_like(d)
    for y in range(h):
        for x in range(w):
            if d[y, x] == 0:
                continue
            win = d[max(0, y - r):y + r + 1, max(0, x - r):x + r + 1]
            yy, xx = np.mgrid[max(0, y - r):min(h, y + r + 1), max(0, x - r):min(w, x + r + 1)]
            ok = win != 0
            wt = np.exp(-((xx - x) ** 2 + (yy - y) ** 2) / (2 * sd * sd)) * np.exp(-(win - d[y, x]) ** 2 / (2 * sr * sr))
            wt, c = wt[ok], win[ok]
            want[y, x] = (wt * c).sum() / wt.sum()
            # weights within 8 u (gd, gr, their product, the argument of gd): the mean moves by <= 2 * 8u * spread;
            # fp32 sums of n terms: n u relative on each, the quotient another u
            u, n = 2.0 ** -24, c.size
            bound[y, x] = 2 * 8 * u * (c.max() - c.min()) + (2 * n + 1) * u * np.abs(c).max()
    assert np.all(np.abs(got - want) <= bound)
    assert np.count_nonzero(got) == np.count_nonzero(d)
