"""Helpers and a random sweep for the label render (``RaycastRGBD.render_labels``, spsg_raycast_labels;
tests/test_gpu_label_render.py).

    python -m tests.fuzz_label_render [cases] [seed]

The label render marches exactly like the forward, and each pixel of a forward's semantic image is its hit voxel's row.
So ``render_labels(labels)`` must equal, bit for bit, ``labels_from_render`` of a forward whose semantic payload is the
one-hot of the labels (C + 1 bins, the last dropped: train.py:590-616), histogram included; a label above C counts as C.
Every case draws C in 1..64, B chunks, F views, an odd or even image size, a grid (the 128x64x64 chunk or a larger one
whose maps do not fit in shared memory), a ray increment, a scene (the synthetic room, or a soup of voxels with random
SDF values), cameras (far, close to a wall, or looking away from the grid), empty chunks, labels (some equal to C, some
above), a debug flag and an index route (int64 rows, packed rows, prebuilt index), and compares the two routes.
"""
import sys

import numpy as np
import torch
import torch.nn.functional as Fn

from spsg_b200 import _native as N
from spsg_b200 import losses
from spsg_b200 import raycast_rgbd_cuda as rc
from spsg_b200 import synthetic as S
from spsg_b200.raycast_rgbd import RaycastRGBD
from tests import fuzz_deterministic as D

BIG_DIMS = (128, 260, 328)  # z, y, x: the march maps of one chunk exceed shared memory (kSmemMaps = false)
DEBUG_FLAGS = (0, N.SPSG_FLAG_NO_CLIP, N.SPSG_FLAG_NO_BRICK_SKIP, N.SPSG_FLAG_SMEM_MAPS, N.SPSG_FLAG_GLOBAL_MAPS)


def module(dev, B, F, w, h, n, C, dims=S.DIMS_ZYX, inc=S.RAY_INCREMENT, flags=0, max_pixels=64):
    m = RaycastRGBD(B, dims, w, h, S.DEPTH_MIN, S.DEPTH_MAX, 50.5 * inc, inc, max_num_frames=F,
                    max_num_locs_per_sample=max(-(-n // B), 1), max_pixels_per_voxel=max_pixels, device=dev,
                    num_classes=C)
    m.flags |= flags
    return m


def voxel_labels(n, C, seed, dev, above=True):
    """(n,) uint8 labels 0..C, a tenth of them C (unlabeled), and with ``above`` a twentieth of them in C+1..255."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    lab = torch.randint(0, C + 1, (n,), generator=g, dtype=torch.int64)
    u = torch.rand(n, generator=g)
    lab[u < 0.1] = C
    if above and C < 255:
        lab[u > 0.95] = torch.randint(C + 1, 256, (int((u > 0.95).sum()),), generator=g)
    return lab.to(torch.uint8).to(dev)


def one_hot_route(m, locs, sdf, labels, view, intr, C):
    """The route the label render replaces: a forward with the one-hot of the labels as semantic payload, then
    labels_from_render of the C-wide image.  Labels above C are first clamped to C (F.one_hot would raise)."""
    n = locs.shape[0]
    onehot = Fn.one_hot(labels.long().clamp(max=C), C + 1)[..., :-1].float().contiguous()
    color = torch.zeros(n, 3, device=sdf.device)
    normal = torch.zeros(n, 3, device=sdf.device)
    with torch.no_grad():
        _, _, _, sem = m(locs, sdf, color, normal, onehot, view, intr)
        lab, hist = losses.labels_from_render(sem, histogram=True)
    torch.cuda.synchronize()
    return lab.clone(), hist.clone()


def cameras(dev, images, rng, w, h, dims, close=0.3, away=0.0):
    """Cameras on a circle around the grid (or 15-25 voxels from a wall of the synthetic room with probability ``close``
    when the grid is the synthetic chunk), and with probability ``away`` cameras that look away from the grid (empty
    views)."""
    if tuple(dims) == tuple(S.DIMS_ZYX):
        view, intr = D.cameras(images, rng, w, h, close)
    else:
        dz, dy, dx = dims
        mats = []
        for _ in range(images):
            az = rng.uniform(0, 2 * np.pi)
            r = rng.uniform(0.6, 1.0) * max(dx, dy)
            eye = (dx / 2 + r * np.cos(az), dy / 2 + r * np.sin(az), dz * rng.uniform(0.6, 1.2))
            mats.append(S.look_at(eye, (dx / 2 + rng.uniform(-20, 20), dy / 2 + rng.uniform(-20, 20), dz * 0.3)))
        view = np.stack(mats).astype(np.float32)
        intr = np.tile(np.asarray(S.INTRINSICS, np.float32), (images, 1))
        intr[:, 0] *= w / S.WIDTH
        intr[:, 2] = (intr[:, 2] + 0.5) * w / S.WIDTH - 0.5
        intr[:, 1] *= h / S.HEIGHT
        intr[:, 3] = (intr[:, 3] + 0.5) * h / S.HEIGHT - 0.5
    for i in range(images):
        if rng.random() < away:
            view[i] = S.look_at((dims[2] / 2, -400.0, dims[0] / 2), (dims[2] / 2, -800.0, dims[0] / 2))
    return torch.from_numpy(np.ascontiguousarray(view, np.float32)).to(dev), torch.from_numpy(intr.astype(np.float32)).to(dev)


def soup(dev, B, dims, seed, count=60000):
    """Voxel soup: ``count`` distinct random cells per chunk inside a box of the grid, SDF values uniform in (-2.95, 2.95) (many
    sign changes, many crossings that fail the threshold or refine onto absent voxels)."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    dz, dy, dx = dims
    lo = (dz // 8, dy // 8, dx // 8)
    hi = (dz * 3 // 4, dy * 7 // 8, dx * 7 // 8)
    box = (hi[0] - lo[0]) * (hi[1] - lo[1]) * (hi[2] - lo[2])
    rows = []
    for b in range(B):
        cells = torch.randperm(box, generator=g)[:min(count, box)]
        z = cells // ((hi[1] - lo[1]) * (hi[2] - lo[2])) + lo[0]
        y = (cells // (hi[2] - lo[2])) % (hi[1] - lo[1]) + lo[1]
        x = cells % (hi[2] - lo[2]) + lo[2]
        rows.append(torch.stack([z, y, x, torch.full_like(z, b)], 1))
    locs = torch.cat(rows).to(torch.int64)
    sdf = (torch.rand(locs.shape[0], 1, generator=g) * 5.9 - 2.95)
    return locs.contiguous().to(dev), sdf.contiguous().to(dev)


def spheres(dev, B, dims, seed):
    """A few spheres and a floor per chunk, the voxels of |sdf| < truncation (torch.nonzero order)."""
    rng = np.random.default_rng(seed)
    dz, dy, dx = dims
    z, y, x = torch.meshgrid(torch.arange(dz, device=dev, dtype=torch.float32),
                             torch.arange(dy, device=dev, dtype=torch.float32),
                             torch.arange(dx, device=dev, dtype=torch.float32), indexing="ij")
    vols = []
    for _ in range(B):
        s = z - 4.0
        for _ in range(int(rng.integers(2, 6))):
            c = (rng.uniform(0.2, 0.8) * dz, rng.uniform(0.2, 0.8) * dy, rng.uniform(0.2, 0.8) * dx)
            r = rng.uniform(0.08, 0.25) * min(dy, dx)
            s = torch.minimum(s, torch.sqrt((z - c[0]) ** 2 + (y - c[1]) ** 2 + (x - c[2]) ** 2) - r)
        vols.append(s)
    sdf = torch.stack(vols)
    idx = torch.nonzero(sdf.abs() < S.TRUNCATION)
    locs = torch.cat([idx[:, 1:], idx[:, :1]], 1).contiguous()
    return locs, sdf[idx[:, 0], idx[:, 1], idx[:, 2], idx[:, 3]].reshape(-1, 1).contiguous()


def scene(dev, B, dims, seed, kind):
    if kind == "room":
        t, n, _ = D.room(dev, B, seed)
        return t["locs"], t["sdf"]
    if kind == "soup":
        return soup(dev, B, dims, seed)
    return spheres(dev, B, dims, seed)


def drop_chunks(locs, sdf, chunks):
    keep = torch.ones(locs.shape[0], dtype=torch.bool, device=locs.device)
    for k in chunks:
        keep &= locs[:, 3] != k
    return locs[keep].contiguous(), sdf[keep].contiguous()


def compare(got, want, what):
    (lab, hist), (wl, wh) = got, want
    assert lab.dtype == torch.uint8 and lab.shape == wl.shape, "%s: shape %s vs %s" % (what, tuple(lab.shape), tuple(wl.shape))
    bad = int((lab != wl).sum())
    assert bad == 0, "%s: %d of %d label pixels differ" % (what, bad, lab.numel())
    assert torch.equal(hist, wh), "%s: histograms differ" % what
    assert torch.equal(hist, torch.bincount(lab.flatten().long(), minlength=hist.numel())), "%s: histogram != labels" % what


def check_case(dev, C, B, F, w, h, seed, dims=S.DIMS_ZYX, kind="room", inc=S.RAY_INCREMENT, flags=0, route="int64",
               empty=(), close=0.3, away=0.0, above=True, n_zero=False):
    """render_labels against the one-hot route on the same voxels and cameras.  Returns the number of pixels hit."""
    rng = np.random.default_rng(seed)
    locs, sdf = scene(dev, B, dims, seed, kind)
    locs, sdf = drop_chunks(locs, sdf, empty)
    if n_zero:
        locs, sdf = locs[:0].contiguous(), sdf[:0].contiguous()
    n = locs.shape[0]
    labels = voxel_labels(n, C, seed + 1, dev, above)
    view, intr = cameras(dev, B * F, rng, w, h, dims, close, away)
    want = one_hot_route(module(dev, B, F, w, h, n, C, dims, inc, flags), locs, sdf, labels, view, intr, C)
    m = module(dev, B, F, w, h, n, C, dims, inc, flags)
    if route == "packed":
        rows = rc.pack_locs_host(locs.cpu(), B, dims).to(dev)
        got = m.render_labels(rows, sdf, labels, view, intr, histogram=True)
    elif route == "prebuilt":
        got = prebuilt_render(m, locs, sdf, labels, view, intr, B, dims)
    else:
        got = m.render_labels(locs, sdf, labels, view, intr, histogram=True)
    torch.cuda.synchronize()
    compare(got, want, "C=%d B=%d F=%d %dx%d dims=%s %s inc=%g flags=%#x %s empty=%s" % (
        C, B, F, w, h, tuple(dims), kind, inc, flags, route, tuple(empty)))
    without = m.render_labels(locs, sdf, labels, view, intr)  # histogram=False: the labels alone, the same
    assert torch.equal(without, got[0])
    return int((got[0] < C).sum())


def prebuilt_render(m, locs, sdf, labels, view, intr, B, dims):
    """The voxel index and SDF brick written by sparsify_predictions(..., raycaster=m) from a dense SDF head that holds
    exactly these rows (rows in torch.nonzero order); the label render must take SPSG_FLAG_INDEX_PREBUILT.  Returns its
    labels and histogram for the rows in the order the caller gave them."""
    from spsg_b200 import sparsify
    outside = torch.full((B, 1) + tuple(dims), 10.0, device=locs.device)
    outside[locs[:, 3], 0, locs[:, 0], locs[:, 1], locs[:, 2]] = sdf[:, 0]
    plocs, psdf = sparsify.sparsify_predictions(outside.contiguous(), S.TRUNCATION, raycaster=m)
    # the labels of the rows in the compaction's order
    dense_lab = torch.zeros((B,) + tuple(dims), dtype=torch.uint8, device=locs.device)
    dense_lab[locs[:, 3], locs[:, 0], locs[:, 1], locs[:, 2]] = labels
    plab = dense_lab[plocs[:, 3], plocs[:, 0], plocs[:, 1], plocs[:, 2]].contiguous()
    seen = []
    real = N.lib.spsg_raycast_labels

    def spy(p, *args):
        seen.append(p._obj.flags)
        return real(p, *args)
    N.lib.spsg_raycast_labels = spy
    try:
        out = m.render_labels(plocs, psdf, plab, view, intr, histogram=True)
    finally:
        N.lib.spsg_raycast_labels = real
    assert plocs.shape[0] == 0 or seen[0] & N.SPSG_FLAG_INDEX_PREBUILT, "the label render did not take the prebuilt index"
    return out


def case(rng):
    C = int(rng.choice([1, 2, 3, 13, 14, 15, 20, 41, 63, 64, int(rng.integers(1, 65))]))
    B = int(rng.choice([1, 2, 3, 8]))
    F = int(rng.choice([1, 2, 3, 5]))
    big = rng.random() < 0.15
    w = int(rng.integers(3, 41)) * 8 + int(rng.integers(0, 8))
    h = int(rng.integers(2, 33)) * 8 + int(rng.integers(0, 8))
    if big:
        B, F, w, h = min(B, 2), min(F, 2), min(w, 160), min(h, 128)
    kind = str(rng.choice(["room", "soup", "spheres"])) if not big else str(rng.choice(["soup", "spheres"]))
    inc = float(rng.choice([S.RAY_INCREMENT, 0.5, 0.37, 1.3]))
    flags = int(rng.choice(DEBUG_FLAGS))
    route = str(rng.choice(["int64", "int64", "packed", "prebuilt"]))
    empty = tuple(int(k) for k in range(B) if B > 1 and rng.random() < 0.2)
    return dict(C=C, B=B, F=F, w=w, h=h, dims=BIG_DIMS if big else S.DIMS_ZYX, kind=kind, inc=inc, flags=flags,
                route=route, empty=empty, close=float(rng.choice([0.0, 0.5])), away=float(rng.choice([0.0, 0.2])),
                n_zero=bool(rng.random() < 0.03), seed=int(rng.integers(1 << 20)))


def run_case(dev, c):
    check_case(dev, c["C"], c["B"], c["F"], c["w"], c["h"], c["seed"], dims=c["dims"], kind=c["kind"], inc=c["inc"],
               flags=c["flags"], route=c["route"], empty=c["empty"], close=c["close"], away=c["away"], n_zero=c["n_zero"])


def sweep(dev, cases, seed):
    rng = np.random.default_rng(seed)
    failures = []
    for _ in range(cases):
        c = case(rng)
        try:
            run_case(dev, c)
        except AssertionError as e:
            failures.append((c, str(e)[:300]))
    return failures


if __name__ == "__main__":
    cases = int(sys.argv[1]) if len(sys.argv) > 1 else 300
    seed = int(sys.argv[2]) if len(sys.argv) > 2 else 0
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    fails = sweep(dev, cases, seed)
    print("label-render sweep: %d cases, %d mismatches" % (cases, len(fails)))
    for f in fails:
        print(f)
    sys.exit(1 if fails else 0)
