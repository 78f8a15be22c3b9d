"""CPU restatement of the depth-frame utilities (csrc/spsg_depth.cu) in numpy.  TEST INFRASTRUCTURE, NOT PRODUCT: it
needs no reference extension, so any shape, sigma or hole pattern has a bit-exact check.  It is anchored to the recorded
reference outputs (tests/golden/ref_pins.json) by tests/test_depth_oracle_cpu.py and tests/test_gpu_depth_oracle.py.

Every float32 operation is the kernel's, in the kernel's order.  Products and sums are numpy float32 operations, which
are correctly rounded like ``__fmul_rn`` / ``__fadd_rn`` / ``__fdiv_rn`` / ``__fsqrt_rn``.  Where nvcc contracts a
product into an FMA (read from the sm_100a SASS: ``sum += weight * cur`` in the bilateral filter, ``1000 * d + 0.5f`` in
the quantisation) or the source writes one (``__fmaf_rn`` in the normals), ``fma32`` computes it with one rounding.

Transcendentals.  The bilateral filter calls ``expf`` (the spatial Gaussian) and ``exp(double)`` (the range Gaussian).
They are not correctly rounded on the device, and numpy's differ from them in the last ulp for some arguments, so the
filter takes them as arguments: ``exp32(x)`` / ``exp64(x)`` map a float32 / float64 array to its exponential in the same
dtype.  The default is numpy's (good to a few ulp: ``bilateral`` with it is compared within a bound); bit-exact
comparisons pass the device's (``torch.exp`` on a CUDA tensor).  The other entry points use no transcendental.

Quantisation of the median fill: ``(int)fl32(1000 d + 0.5)``, one rounding, then PTX ``cvt.rzi.s32.f32``: truncation
towards zero, saturating at the int32 range, NaN -> 0 (numpy's float -> int cast is undefined there, so ``quantise``
spells these cases out).
"""
import numpy as np

F32 = np.float32
FILL_RADIUS = 5           # kFillRadius: the median window is 11 x 11
TABLE_RADIUS = 8          # kTableRadius: radii above it compute the spatial Gaussian per tap (same values)
MAX_FILL_ROUNDS = 64      # SPSG_DEPTH_MAX_FILL_ROUNDS


def np_exp(x):
    return np.exp(x)


def fma32(a, b, c):
    """fl32(a * b + c) with one rounding, elementwise on float32 inputs.  The product of two float32 values is exact in
    float64; TwoSum gives the exact error of the float64 sum; rounding that sum to odd and then to float32 is correctly
    rounded (53 >= 2 * 24 + 2)."""
    a, b, c = (np.asarray(v, F32).astype(np.float64) for v in (a, b, c))
    with np.errstate(all="ignore"):
        p = a * b
        s = p + c
        bb = s - p
        err = (p - (s - bb)) + (c - bb)
        even = (s.view(np.int64) & 1) == 0
        bump = np.isfinite(s) & (err != 0) & even
        s = np.where(bump, np.nextafter(s, np.where(err > 0, np.inf, -np.inf)), s)
        return s.astype(F32)


def _frames(depth):
    d = np.ascontiguousarray(depth, F32)
    return d.reshape((-1,) + d.shape[-2:])


def valid(d):
    """depth_valid: neither 0 (either sign) nor -inf.  NaN and +inf are valid."""
    return (d != 0) & (d != -np.inf)


def bilateral(depth, sigma_d, sigma_r, exp32=np_exp, exp64=np_exp):
    """bilateral_tile on (B, 1, H, W) or (B, H, W) depth; same shape out.  Radius ceil(2 sigma_d) in double; offsets
    x outer, y inner; out-of-frame and invalid taps skipped; gd = expf(fl32(-fl32(dx^2 + dy^2) / fl32(fl32(2 sd) sd))),
    gr = fl32(exp(-fl32(dist^2) / ((2 sr) sr)) in double); weight = gd gr; sum_weight += weight; sum = fma(weight, cur,
    sum); result sum / sum_weight if sum_weight > 0, else 0; an invalid centre gives 0."""
    shape = np.shape(depth)
    d = _frames(depth)
    b, h, w = d.shape
    sd, sr = F32(sigma_d), F32(sigma_r)
    r = int(np.ceil(2.0 * np.float64(sd)))
    offs = np.arange(-r, r + 1)
    dx2 = (offs[:, None] ** 2 + offs[None, :] ** 2).astype(F32)             # [dx + r, dy + r]
    gd = np.asarray(exp32(-(dx2 / ((sd + sd) * sd))), F32)
    sr2 = (np.float64(sr) + np.float64(sr)) * np.float64(sr)
    pad = np.zeros((b, h + 2 * r, w + 2 * r), F32)                           # 0 = invalid: out-of-frame taps are skipped
    pad[:, r:r + h, r:r + w] = d
    s = np.zeros_like(d)
    sw = np.zeros_like(d)
    with np.errstate(all="ignore"):
        for i, dx in enumerate(offs):
            # the range Gaussians of one column of offsets in one exp64 call
            dist = np.stack([pad[:, r + dy:r + dy + h, r + dx:r + dx + w] for dy in offs]) - d
            grs = np.asarray(exp64((-(dist * dist)).astype(np.float64) / sr2), np.float64).astype(F32)
            for j, dy in enumerate(offs):
                cur = pad[:, r + dy:r + dy + h, r + dx:r + dx + w]
                ok = valid(cur)
                weight = gd[i, j] * grs[j]
                sw = np.where(ok, sw + weight, sw)
                s = np.where(ok, fma32(weight, cur, s), s)
        out = np.where(valid(d) & (sw > 0), s / np.where(sw > 0, sw, F32(1)), F32(0)).astype(F32)
    return out.reshape(shape)


def quantise(d):
    """(int)(1000 * d + 0.5f) as the kernel computes it: fl32 of the exact value, then cvt.rzi.s32.f32."""
    x = fma32(F32(1000), d, F32(0.5)).astype(np.float64)
    q = np.trunc(np.nan_to_num(x, nan=0.0, posinf=2.0 ** 31, neginf=-2.0 ** 31))
    return np.clip(q, -2 ** 31, 2 ** 31 - 1).astype(np.int64)


def median_value(qs):
    """The order statistic of one window's quantised valid depths: the ((n+1)/2)-th smallest, 0-based, 0 for n < 2."""
    qs = np.sort(np.asarray(qs, np.int64))
    return int(qs[(qs.size + 1) // 2]) if qs.size >= 2 else 0


def dequantise(val):
    """A hole's value from its window's order statistic: 0 if val <= 0, else fl32(0.001f * fl32(val))."""
    val = np.asarray(val, np.int64)
    return np.where(val <= 0, F32(0), F32(0.001) * val.astype(F32)).astype(F32)


def median_fill(depth, chunk=1 << 15):
    """median_fill_tile on (B, 1, H, W) or (B, H, W) depth; same shape out.  Valid pixels are copied; a hole (0 or -inf)
    takes dequantise(median_value(window)) over the valid pixels of its 11 x 11 window that lie in the frame."""
    shape = np.shape(depth)
    d = _frames(depth)
    b, h, w = d.shape
    R, D = FILL_RADIUS, 2 * FILL_RADIUS + 1
    ok = np.zeros((b, h + 2 * R, w + 2 * R), bool)
    ok[:, R:R + h, R:R + w] = valid(d)
    q = np.zeros(ok.shape, np.int64)
    q[:, R:R + h, R:R + w] = quantise(d)
    out = d.copy()
    hb, hy, hx = np.nonzero(~valid(d))
    wy, wx = np.divmod(np.arange(D * D), D)
    big = np.iinfo(np.int64).max                                             # sorts after every int32 value
    for s in range(0, hb.size, chunk):
        bb, yy, xx = hb[s:s + chunk, None], hy[s:s + chunk, None] + wy, hx[s:s + chunk, None] + wx
        m = ok[bb, yy, xx]
        n = m.sum(1)
        vals = np.sort(np.where(m, q[bb, yy, xx], big), axis=1)
        k = np.minimum((n + 1) // 2, D * D - 1)
        val = np.where(n >= 2, vals[np.arange(n.size), k], 0)
        out[hb[s:s + chunk], hy[s:s + chunk], hx[s:s + chunk]] = dequantise(val)
    return out.reshape(shape)


def camspace(depth, intr):
    """camera_point of every pixel: depth (B, 1, H, W) or (B, H, W), intrinsics (B, 4) = fx, fy, mx, my per frame ->
    (B, H, W, 3).  (x, y) = (fl32(d fl32(fl32(x - mx) / fx)), fl32(d fl32(fl32(y - my) / fy))), z = d; d == 0 -> 0."""
    d = _frames(depth)
    b, h, w = d.shape
    k = np.ascontiguousarray(intr, F32).reshape(-1, 4)[:b]
    fx, fy, mx, my = (k[:, i, None, None] for i in range(4))
    with np.errstate(all="ignore"):
        px = (np.arange(w, dtype=F32)[None, None, :] - mx) / fx
        py = (np.arange(h, dtype=F32)[None, :, None] - my) / fy
        out = np.stack(np.broadcast_arrays(d * px, d * py, d), -1).astype(F32)
    out[d == 0] = 0
    return out


def normals(cam):
    """normal_from_points at every interior pixel of (B, H, W, 3) camera-space images; border pixels 0.  Gate: some of
    the five points' x non-zero and none -inf.  a = pc - mc, b = cp - cm; n = (fma(ay, bz, -(az by)), fma(az, bx, -(ax bz)),
    fma(ax, by, -(ay bx))); l = sqrt(fma(nz, nz, fma(ny, ny, nx nx))); n / -l where l > 0, else 0."""
    c = np.ascontiguousarray(cam, F32)
    out = np.zeros_like(c)
    if c.shape[1] < 3 or c.shape[2] < 3:
        return out
    cc, pc, cp, mc, cm = c[:, 1:-1, 1:-1], c[:, 2:, 1:-1], c[:, 1:-1, 2:], c[:, :-2, 1:-1], c[:, 1:-1, :-2]
    xs = [p[..., 0] for p in (cc, pc, cp, mc, cm)]
    gate = np.logical_or.reduce([x != 0 for x in xs]) & np.logical_and.reduce([x != -np.inf for x in xs])
    with np.errstate(all="ignore"):
        a, bv = pc - mc, cp - cm
        ax, ay, az = a[..., 0], a[..., 1], a[..., 2]
        bx, by, bz = bv[..., 0], bv[..., 1], bv[..., 2]
        nx, ny, nz = fma32(ay, bz, -(az * by)), fma32(az, bx, -(ax * bz)), fma32(ax, by, -(ay * bx))
        l = np.sqrt(fma32(nz, nz, fma32(ny, ny, nx * nx)))
        n = np.stack([nx / -l, ny / -l, nz / -l], -1)
    out[:, 1:-1, 1:-1] = np.where((gate & (l > 0))[..., None], n, F32(0))
    return out


def depth2normals(depth, intr, max_fill_iters=40, exp32=np_exp, exp64=np_exp, sigma_d=2.0, sigma_r=0.1):
    """Depth2Normals.forward (spsg_depth_to_normals): filter, then max_fill_iters // 2 rounds of depth <- fill(filtered),
    filtered <- fill(depth), stopping before a round when no zero is left; camera space and normals of the filled depth.

    Returns a dict: ``depth`` (the filled frame, what the caller's tensor holds afterwards), ``filtered``, ``camspace``,
    ``normals`` (B, H, W, 3, computed in any case), ``hole_counts`` (int32, MAX_FILL_ROUNDS + 1: [0] the zeros of the
    input, [r] the zeros after round r, 0 past the round that left none) and ``none`` (forward returns None: a budget
    above 0 whose last round left zeros, or whose input had zeros when it allows no round)."""
    shape = np.shape(depth)
    d = _frames(depth).copy()
    filt = bilateral(d, sigma_d, sigma_r, exp32, exp64)
    counts = np.zeros(MAX_FILL_ROUNDS + 1, np.int32)
    counts[0] = np.count_nonzero(d == 0)
    rounds = max_fill_iters // 2
    for r in range(rounds):
        if counts[r] == 0:
            break
        d = median_fill(filt)
        counts[r + 1] = np.count_nonzero(d == 0)
        filt = median_fill(d)
    cam = camspace(d, intr)
    return {"depth": d.reshape(shape), "filtered": filt.reshape(shape), "camspace": cam, "normals": normals(cam),
            "hole_counts": counts, "none": max_fill_iters > 0 and counts[rounds] != 0}


class Module:
    """The four entry points of ``depth_utils_cuda`` with its signatures, on CPU torch tensors, writing their outputs in
    place: a stand-in for the extension that ``oracle.ref_pins.PinnedModule`` can check against the recorded outputs."""

    def __init__(self, exp32=np_exp, exp64=np_exp):
        self.exp32, self.exp64 = exp32, exp64

    @staticmethod
    def _put(out, a):
        import torch
        out.copy_(torch.from_numpy(np.ascontiguousarray(a)).view(out.shape))

    def bilateral_filter_floatmap(self, out, depth, sigma_d, sigma_r):
        self._put(out, bilateral(depth.numpy(), sigma_d, sigma_r, self.exp32, self.exp64))

    def median_fill_depthmap(self, out, depth):
        self._put(out, median_fill(depth.numpy()))

    def convert_depth_to_cameraspace(self, out, depth, intr, depth_min, depth_max):
        self._put(out, camspace(depth.numpy(), intr.numpy()))

    def compute_normals(self, out, cam):
        self._put(out, normals(cam.numpy()))


def bits(a):
    """int32 view of a float32 array with every NaN as 0x7fffffff: the device writes the canonical NaN where x86
    propagates payloads, so NaN outputs are compared as NaN, everything else bit for bit."""
    a = np.ascontiguousarray(a, F32)
    return np.where(np.isnan(a), np.int32(0x7fffffff), a.view(np.int32))


# --- random inputs for the randomised checks (tests/test_gpu_depth_oracle.py, tests/fuzz_depth.py) ---------------------

SPECIALS = (-np.inf, np.nan, np.inf)


def random_frames(rng, b, h, w, holes=None, specials=None):
    """(B, 1, H, W) float32 depth: a smooth surface with noise, a random share of zero pixels, maybe a hole block, and
    maybe a sprinkle of -inf / NaN / +inf, sub-millimetre, negative (q = -1 included) pixels."""
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float64)
    d = np.stack([rng.uniform(0.5, 4) + 0.01 * rng.uniform(-1, 1) * xx + 0.01 * rng.uniform(-1, 1) * yy +
                  0.2 * np.sin(xx / rng.uniform(3, 20)) * np.cos(yy / rng.uniform(3, 20)) +
                  0.02 * rng.standard_normal((h, w)) for _ in range(b)])
    d = np.maximum(d, 0.05)
    if rng.random() < 0.1:
        d *= rng.uniform(0.001, 20, d.shape)                                   # windows spanning metres
    holes = rng.uniform(0, 0.6) if holes is None else holes
    d[rng.random(d.shape) < holes] = 0.0
    if rng.random() < 0.5:
        y0, x0 = int(rng.integers(0, h)), int(rng.integers(0, w))
        d[:, y0:y0 + int(rng.integers(1, 30)), x0:x0 + int(rng.integers(1, 30))] = 0.0
    if specials if specials is not None else rng.random() < 0.5:
        pick = rng.random(d.shape) < rng.uniform(0.005, 0.05)
        kinds = rng.integers(0, 6, d.shape)
        neg = -rng.uniform(0.0015, 0.0025, d.shape)                            # q = -1 (and its two edges)
        val = np.select([kinds < 3, kinds == 3, kinds == 4],
                        [np.array(SPECIALS)[np.minimum(kinds, 2)], rng.uniform(0, 6e-4, d.shape), neg],
                        -rng.uniform(0, 3, d.shape))
        val = np.where((kinds == 2) & (rng.random(d.shape) < 0.8), -np.inf, val)   # +inf rarely
        d = np.where(pick, val, d)
    return d.astype(F32)[:, None]


def random_intrinsics(rng, b, h, w):
    """(B, 4) float32: fx, fy, mx, my different for every frame."""
    return np.stack([rng.uniform(50, 300, b), rng.uniform(50, 300, b), w / 2 - 0.5 + rng.uniform(-5, 5, b),
                     h / 2 - 0.5 + rng.uniform(-5, 5, b)], 1).astype(F32)


def random_case(rng):
    """One randomised case: shape (down to 1 x 1), frames, intrinsics, bilateral sigmas, fill budget."""
    if rng.random() < 0.25:
        b, h, w = int(rng.integers(1, 4)), int(rng.integers(1, 12)), int(rng.integers(1, 40))
    else:
        b, h, w = int(rng.integers(1, 4)), int(rng.integers(8, 120)), int(rng.integers(8, 160))
    sigma_d = float(rng.choice([0.3, 2.0, 2.3, 4.0, 4.01, float(rng.uniform(0.2, 5.5))]))
    sigma_r = float(np.exp(rng.uniform(np.log(0.01), np.log(1.0))))
    iters = int(rng.choice([0, 1, 2, 3, 4, 40, 128]))
    return (random_frames(rng, b, h, w), random_intrinsics(rng, b, h, w), sigma_d, sigma_r, iters)
