"""Float64 oracle of the raycast backward's per-voxel gather, built from a forward's renderings alone.  TEST
INFRASTRUCTURE, NOT PRODUCT: it needs no reference extension, so any new shape, table size or flag combination has a
backward check.

Pixel -> voxel map.  The caller writes the voxel id into the normal payload, which no loss reads:
``vals_normals[v] = (v + 1, 0.5, -0.25)`` (exact in fp32 for N < 2^24; the forward copies a non-zero normal verbatim).  A
hit pixel is one whose depth is not -inf; its voxel is ``normal[..., 0] - 1``.  ``pixel_map`` checks that the colour and
semantic renderings of every hit pixel equal that voxel's payload bit for bit, and that every miss is -inf in all four.

Registration tables.  For a voxel v and a view f (image ``locs[v, 3] * F + f``), ``check_tables`` requires
``mapping3dto2d_num[f*N + v]`` to equal the number of pixels of v in that image exactly, and the first
``min(num, max_pix)`` table entries to be distinct pixels of v.  The pixel set S(v, f) the gather averages over is then
exactly those entries: all of v's pixels when ``num <= max_pix``, the table's subset when the voxel overflowed it.  That
subset is the only input taken from the kernel under test, and it has been validated.

Reference: ``d[v] = sum_f sum_{p in S(v,f)} G[p] / |S(v,f)|``, 21 channels routed as the kernel routes them (0-13
semantic, 14-16 colour, 17 depth -> sdf, 18-20 normal), in float64.

Per-entry bounds, from the kernel's arithmetic (spsg_backward.cuh, backward_gather_kernel).  u = 2^-24.
  * One view: the kernel sums the fp32 rows in double (error <= (cnt-1) 2^-53 sum|g|), multiplies by
    ``fl32(1/cnt)`` (``__frcp_rn``: relative u) in double (relative 2^-53) and rounds once to fp32 (relative u).  With
    cnt <= 256: ``|err| <= 2^-23 |m| + 2^-45 sum|g| / cnt`` for the exact mean m (the double-precision terms are inside the
    second term, since |m| <= sum|g| / cnt).  Results below the fp32 normal range may be flushed to 0: add 2^-126.
  * Several views, float atomics (any order) onto a cleared row: each view's mean as above, plus the F - 1 fp32
    additions: ``(F - 1) u sum_f |m_f|``.
  * Several views, deterministic (``SPSG_FLAG_DETERMINISTIC_GRADS``): the kernel computes
    ``tot = 0f; for f in view order: tot = fl32(tot + fl32(S_f * fl64(fl32(1/cnt_f))))`` with S_f its double sum.  The
    oracle does the same with its own double sum S'_f, |S_f - S'_f| <= 2 cnt 2^-53 sum|g|: both round to the same fp32
    value unless the double product lies within that distance (plus two double roundings) of an fp32 rounding boundary.
    Such entries are flagged as near-ties and excluded (and counted); every other entry must match bit for bit.
  * Fused 2D losses: each pixel's gradient row is recomputed in fp32 by the kernel, so ``fused_pixel_grads`` returns a
    per-pixel bound image that the gather propagates (``sum_p b[p] / cnt``).  The semantic row uses ``__expf`` of
    ``fl32(l_k - max)``: the argument's rounding and ``ex2.approx``'s scaling by log2(e) cost about 3 |x| u relative (x =
    l_k - max <= 0), which exceeds the 2^-21 of ``ex2.approx`` for |x| > 2 -- harmless only because those terms carry a
    factor e^x.  ``ex2.approx.ftz`` flushes exponentials below 2^-126 to 0 (an absolute |f| 2^-120 per channel), and
    the fused row flushes products below 2^-126 to 0 (an absolute 2^-126 per channel).
The gather's own terms are never looser than 1e-5 of the entry's sum of magnitudes (``sum_f sum_p |g| / cnt``; for the
semantic target channel both summands of ``f s_y - f`` count); ``gather`` asserts it.  Propagated per-pixel bounds are
below 1e-5 of the pixel's magnitudes too, except for the exponent term and the ftz floor above.
"""
import numpy as np

U = 2.0 ** -24
NINF = -np.inf


def voxel_normals(n):
    """(N, 3) fp32 normal payload carrying the voxel id: (v + 1, 0.5, -0.25)."""
    assert n < (1 << 24)
    out = np.empty((n, 3), np.float32)
    out[:, 0] = np.arange(1, n + 1, dtype=np.float32)
    out[:, 1] = 0.5
    out[:, 2] = -0.25
    return out


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.int32)


def pixel_map(color, depth, normal, semantic, vals_color, vals_semantic):
    """Renderings (I,H,W,3) / (I,H,W) / (I,H,W,3) / (I,H,W,14) as numpy fp32 -> (I, H*W) int64 voxel id, -1 = miss.
    Asserts the payload identities described in the module docstring."""
    n = vals_color.shape[0]
    i = depth.shape[0]
    depth = depth.reshape(i, -1)
    color, normal, semantic = color.reshape(i, -1, 3), normal.reshape(i, -1, 3), semantic.reshape(i, -1, 14)
    hit = depth != NINF
    assert not np.isnan(depth).any(), "NaN depth"
    miss = ~hit
    for name, img in (("colour", color), ("normal", normal), ("semantic", semantic)):
        assert bool((img[miss] == NINF).all()), "a miss pixel has a finite %s" % name
    vid = normal[..., 0].astype(np.float64) - 1.0
    vox = np.where(hit, vid, -1.0)
    assert bool((vox[hit] == np.round(vox[hit])).all()) and bool(((vox[hit] >= 0) & (vox[hit] < n)).all()), \
        "hit pixel without a valid voxel id in its normal"
    vox = vox.astype(np.int64)
    v = vox[hit]
    assert bool((normal[hit][:, 1] == 0.5).all() and (normal[hit][:, 2] == -0.25).all()), "normal payload altered"
    assert bool((_bits(color[hit]) == _bits(vals_color[v])).all()), "colour of a hit pixel is not its voxel's payload"
    assert bool((_bits(semantic[hit]) == _bits(vals_semantic[v])).all()), "semantic of a hit pixel is not its payload"
    return vox


class Tables:
    """The validated pixel sets S(v, f) as flat pairs: ``row`` (= f*N + v) and ``gpix`` (global pixel index
    image*P + p), with per-row ``cnt`` = |S(v, f)|; ``overflow`` = rows whose voxel had more pixels than the table."""

    def __init__(self, n, views, row, gpix, cnt, overflow):
        self.n, self.views, self.row, self.gpix, self.cnt, self.overflow = n, views, row, gpix, cnt, overflow


def check_tables(vox, mapping, num, chunk, views):
    """vox: (I, P) from ``pixel_map``; mapping (F*N, max_pix) int32; num (>= F*N,) int32; chunk (N,) = locs[:, 3]."""
    n = chunk.shape[0]
    images, P = vox.shape
    max_pix = mapping.shape[1]
    num = num[:views * n].astype(np.int64)
    # pixels per (voxel, view) from the renderings
    img_of = np.repeat(np.arange(images), P).reshape(images, P)
    hit = vox >= 0
    v_hit, i_hit = vox[hit], img_of[hit]
    assert bool((i_hit // views == chunk[v_hit]).all()), "a voxel was rendered into another chunk's image"
    rows_hit = (i_hit % views) * n + v_hit
    count = np.bincount(rows_hit, minlength=views * n)
    bad = np.nonzero(count != num)[0]
    assert bad.size == 0, "mapping3dto2d_num differs from the rendered pixel counts at %d rows (first: row %d has %d, " \
        "rendered %d)" % (bad.size, bad[0], num[bad[0]], count[bad[0]])
    rows = np.nonzero(num > 0)[0]
    k = np.minimum(num[rows], max_pix)
    ent = mapping[:views * n][rows].astype(np.int64)
    used = np.arange(max_pix)[None, :] < k[:, None]
    assert bool(((ent >= 0) & (ent < P))[used].all()), "table entry outside the image"
    srt = np.sort(np.where(used, ent, P + np.arange(max_pix)[None, :]), axis=1)
    assert bool((np.diff(srt, axis=1) != 0).all()), "a pixel is registered twice for one (voxel, view)"
    v = rows % n
    image = chunk[v] * views + rows // n
    rr = np.repeat(rows, k)
    pix = ent[used]
    ii = np.repeat(image, k)
    assert bool((vox[ii, pix] == rr % n).all()), "a table entry is a pixel of another voxel"
    cnt = np.zeros(views * n, np.int64)
    cnt[rows] = k
    return Tables(n, views, rr, ii * P + pix, cnt, rows[num[rows] > max_pix])


def _rowsum(tab, x):
    """Per-row sums of per-pixel values x (num_pixels, C) over S, float64 -> (F*N, C)."""
    out = np.zeros((tab.views * tab.n, x.shape[1]))
    xs = x[tab.gpix]
    for c in range(x.shape[1]):
        out[:, c] = np.bincount(tab.row, weights=xs[:, c], minlength=tab.views * tab.n)
    return out


def near_tie(x, delta):
    """True where float64 x lies within delta of an fp32 rounding boundary."""
    r = x.astype(np.float32)
    r64 = r.astype(np.float64)
    up = np.nextafter(r, np.float32(np.inf)).astype(np.float64)
    dn = np.nextafter(r, np.float32(-np.inf)).astype(np.float64)
    with np.errstate(invalid="ignore"):
        dist = np.minimum(np.abs(x - (r64 + up) / 2), np.abs(x - (r64 + dn) / 2))
    return dist <= delta


class Gather:
    """want / bound / mag: (N, 21) float64; exact: (N, 21) fp32 emulation of the deterministic kernel or None;
    ties: its excluded entries."""


def gather(tab, G, pixel_bound=None, mag=None, deterministic=False):
    """G: (num_pixels, 21) per-pixel gradients (float64; fp32 values for the plain backward).  pixel_bound: per-pixel
    error bound of the kernel's recomputed rows (fused), None = the rows are G exactly.  mag: per-pixel magnitudes
    (default |G|).  deterministic: also the bit-exact fp32 emulation (plain rows only)."""
    n, F = tab.n, tab.views
    G = np.asarray(G, np.float64)
    mag = np.abs(G) if mag is None else mag
    S = _rowsum(tab, G)
    A = _rowsum(tab, mag)
    Bp = _rowsum(tab, pixel_bound) if pixel_bound is not None else np.zeros_like(S)
    cnt = tab.cnt[:, None].astype(np.float64)
    live = cnt > 0
    c1 = np.where(live, cnt, 1.0)
    m = np.where(live, S / c1, 0.0)
    per = np.where(live, 2.0 ** -23 * (np.abs(m) + Bp / c1) + 2.0 ** -45 * A / c1 + Bp / c1 + 2.0 ** -126, 0.0)
    r = lambda x: x.reshape(F, n, 21).sum(0)
    out = Gather()
    out.want = r(m)
    out.mag = r(np.where(live, A / c1, 0.0))
    out.bound = r(per) + (F - 1) * U * r(np.abs(m) + np.where(live, Bp / c1, 0.0))
    own = r(np.where(live, 2.0 ** -23 * np.abs(m) + 2.0 ** -45 * A / c1, 0.0)) + (F - 1) * U * r(np.abs(m))
    assert bool((own <= 1e-5 * out.mag + 2.0 ** -126).all()), "gather bound looser than 1e-5"
    out.exact, out.ties = None, None
    if deterministic:
        assert pixel_bound is None
        inv = np.where(live, (1.0 / c1).astype(np.float32).astype(np.float64), 0.0)
        x = S * inv
        delta = 2 * cnt * 2.0 ** -53 * A * inv + 2.0 ** -51 * np.abs(x)
        tie = live & near_tie(x, delta)
        y = x.astype(np.float32).reshape(F, n, 21)
        tot = np.zeros((n, 21), np.float32)
        for f in range(F):
            tot = np.where(live.reshape(F, n, 1)[f], tot + y[f], tot)
        out.exact = tot
        out.ties = tie.reshape(F, n, 21).any(0)
    return out


def route(d_semantic, d_color, d_depth, d_normal):
    """The four gradient buffers (rows [0, N)) as the kernel's 21 channels, float64."""
    return np.concatenate([d_semantic.reshape(-1, 14), d_color.reshape(-1, 3), d_depth.reshape(-1, 1),
                           d_normal.reshape(-1, 3)], 1).astype(np.float64)


def unroute(x):
    """(N, 21) -> (sdf, colour, normal, semantic) in the order the autograd Functions return them."""
    return x[:, 17:18], x[:, 14:17], x[:, 18:21], x[:, 0:14]


def plain_pixel_grads(grad_color, grad_depth, grad_normal, grad_semantic):
    """Upstream gradient images -> (num_pixels, 21) in the kernel's channel order."""
    return route(grad_semantic, grad_color, grad_depth, grad_normal)


def compare(got, g, what="", exact=False):
    """got: (N, 21) fp32 of the kernel.  Raises AssertionError on the first failing entries.  Returns the number of
    near-tie entries excluded (exact mode)."""
    got = np.asarray(got, np.float32)
    assert not np.isnan(got).any(), "%s: NaN in the voxel gradients (%d entries)" % (what, int(np.isnan(got).sum()))
    if exact:
        bad = (_bits(got) != _bits(g.exact)) & ~g.ties
        if bad.any():
            v, c = np.argwhere(bad)[0]
            raise AssertionError("%s: %d entries differ from the fp32 emulation bit for bit (first voxel %d channel %d: "
                                 "%r vs %r)" % (what, int(bad.sum()), v, c, got[v, c], g.exact[v, c]))
        return int(g.ties.sum())
    err = np.abs(got.astype(np.float64) - g.want)
    bad = ~(err <= g.bound)
    if bad.any():
        v, c = np.argwhere(bad)[0]
        raise AssertionError("%s: %d entries outside their bound (first voxel %d channel %d: got %r want %r, err %.3g, "
                             "bound %.3g, magnitude %.3g)" % (what, int(bad.sum()), v, c, float(got[v, c]),
                                                               g.want[v, c], err[v, c], g.bound[v, c], g.mag[v, c]))
    return 0


# ---------------------------------------------------------------------------------------------------------------------
# Fused 2D losses: the upstream images of the three terms (oracle/losses_ref.py), differentiated by hand in float64
# ---------------------------------------------------------------------------------------------------------------------

def fused_pixel_grads(color, depth, semantic, target_depth=None, target_color=None, weight_color=None, label=None,
                      class_weight=None, voxelsize=0.02, weights=(1.0, 1.0, 1.0), grad_scale=1.0, upstream=None):
    """Renderings (fp32 numpy, any leading shape) and targets -> (G, mag, bound, loss) where G, mag and bound are
    (num_pixels, 21) float64 and loss = (values[4], bounds[4]): the depth / colour / semantic terms and the weighted total.
    The discrete decisions (validity, signs, label < 14) are taken on the fp32 expressions, as torch takes them.
    upstream: (grad_color, grad_depth, grad_normal, grad_semantic) fp32 images or None each, added in fp32."""
    P = depth.size
    r = depth.reshape(P).astype(np.float32)
    c = color.reshape(P, 3).astype(np.float32)
    lg = semantic.reshape(P, 14).astype(np.float32)
    wd, wc, ws = (float(np.float32(x)) for x in weights)  # the kernel's weights are fp32
    grad_scale = float(np.float32(grad_scale))
    vs32 = np.float32(voxelsize)
    G = np.zeros((P, 21))
    mag = np.zeros((P, 21))
    bnd = np.zeros((P, 21))
    vals, lb = [0.0, 0.0, 0.0], [0.0, 0.0, 0.0]
    if target_depth is not None:
        td = target_depth.reshape(P).astype(np.float32)
        valid = (r != NINF) & (td != 0)
        with np.errstate(invalid="ignore", over="ignore"):
            d32 = np.where(valid, r * vs32 - td, np.float32(0))
        cntd = float(valid.sum())
        g = np.sign(d32).astype(np.float64) * wd * float(vs32) * grad_scale / cntd if cntd else np.zeros(P)
        G[:, 17] = g
        bnd[:, 17] = 4 * U * np.abs(g)
        rv = np.where(valid, r, 0).astype(np.float64) * float(vs32)
        d64 = np.abs(rv - np.where(valid, td, 0))
        vals[0] = d64.sum() / cntd if cntd else np.nan
        lb[0] = ((2 * U * (np.abs(rv) + np.abs(np.where(valid, td, 0)))).sum() + 33 * U * d64.sum()) / cntd + U * vals[0] \
            if cntd else 0.0
    if target_color is not None:
        tc = target_color.reshape(P, 3).astype(np.float32)
        w32 = np.ones(P, np.float32) if weight_color is None else weight_color.reshape(P).astype(np.float32)
        valid = c != NINF
        with np.errstate(invalid="ignore", over="ignore"):
            d32 = np.where(valid, c * w32[:, None] - tc * w32[:, None], np.float32(0))
        cntc = float(valid.sum())
        g = np.sign(d32).astype(np.float64) * w32[:, None] * wc * grad_scale / cntc if cntc else np.zeros((P, 3))
        G[:, 14:17] = g
        bnd[:, 14:17] = 4 * U * np.abs(g)
        cw64 = np.where(valid, c, 0).astype(np.float64) * w32[:, None]
        tw64 = np.where(valid, tc, 0).astype(np.float64) * w32[:, None]
        d64 = np.abs(cw64 - tw64)
        vals[1] = d64.sum() / cntc if cntc else np.nan
        lb[1] = ((3 * U * (np.abs(cw64) + np.abs(tw64))).sum() + 35 * U * d64.sum()) / cntc + U * vals[1] if cntc else 0.0
    if label is not None:
        y = label.reshape(P).astype(np.int64)
        valid = (y < 14) & (lg[:, 0] != NINF)
        cwt = np.ones(14) if class_weight is None else class_weight.astype(np.float32).astype(np.float64)
        l64 = np.where(valid[:, None], lg, 0).astype(np.float64)
        mx = l64.max(1)
        x = l64 - mx[:, None]
        e = np.exp(x)
        s = e.sum(1)
        sm = e / s[:, None]
        yv = np.where(valid, y, 0)
        w = np.where(valid, cwt[yv], 0.0)
        sw = w.sum()
        onehot = np.zeros((P, 14))
        onehot[np.arange(P), yv] = 1.0
        f = ws * grad_scale * w / sw if sw else np.zeros(P)
        G[:, :14] = np.where(valid[:, None], f[:, None] * (sm - onehot), 0.0)
        # per-pixel bound (module docstring): exp terms, their fp32 sum, the factor chain, the final rounding
        eps_k = (3 * np.abs(x) + 2) * U + 2.0 ** -21
        eps_sum = 14 * U + (sm * eps_k).sum(1)
        eps_f = (34 + 5) * U  # normaliser: 32-lane fp32 sum + its rounding; then w*scale/norm, *w, *rcp
        af = np.abs(f)[:, None]
        b = af * (sm * (eps_k + eps_sum[:, None] + U) + eps_f * (sm + onehot) + U * np.abs(sm - onehot)) + \
            af * 2.0 ** -120 + 2.0 ** -126
        bnd[:, :14] = np.where(valid[:, None], b, 0.0)
        mag[:, :14] = np.where(valid[:, None], af * (sm + onehot), 0.0)
        nll = np.log(s) - x[np.arange(P), yv]
        vals[2] = (w * nll).sum() / sw if sw else np.nan
        ep = w * (2.0 ** -20 + eps_sum + 2.0 ** -23 * (np.log(s) + np.abs(mx) + np.abs(l64[np.arange(P), yv]))) + U * w * nll
        lb[2] = (ep.sum() + 33 * U * (w * nll).sum()) / sw + (34 + 2) * U * abs(vals[2]) if sw else 0.0
    mag[:, 14:18] = np.abs(G[:, 14:18])
    if upstream is not None:
        gsum = np.zeros((P, 21))
        for u, sl in zip(upstream, (slice(14, 17), slice(17, 18), slice(18, 21), slice(0, 14))):
            if u is not None:
                gsum[:, sl] = u.reshape(P, sl.stop - sl.start).astype(np.float32)
        have = gsum != 0
        bnd = np.where(have, bnd + U * (np.abs(G) + np.abs(gsum) + bnd), bnd)
        G = G + gsum
        mag = mag + np.abs(gsum)
    w3 = (wd, wc, ws)
    present = (target_depth is not None, target_color is not None, label is not None)
    total = sum(wi * v for wi, v, p in zip(w3, vals, present) if p)
    tb = sum(abs(wi) * b + 3 * U * abs(wi * v) for wi, v, b, p in zip(w3, vals, lb, present) if p) + U * abs(total)
    return G, mag, bnd, (vals + [total], lb + [tb])
