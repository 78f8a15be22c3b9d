"""Randomised sweep of deterministic mode (SPSG_FLAG_DETERMINISTIC); tests/test_gpu_deterministic.py runs a seeded slice
under pytest and uses the same helpers.

Each case renders random chunks of the synthetic room (B = 1-8, F = 1-5, max_pixels_per_voxel 1-64) from random cameras,
close ones (0.3-0.5 m from a wall, where most (voxel, view) rows overflow their table) mixed with far ones, with random
schedule flags, and checks:
  * tables against the renderings: the voxel id sits in the normal payload, so every pixel's voxel is known; row (v, f) must
    hold sorted(S(v, f))[:P] exactly, and its count |S(v, f)|;
  * schedule independence: the same case with the deterministic flag and each of {0, SMEM_MAPS, GLOBAL_MAPS,
    NO_BRICK_SKIP, NO_CLIP} gives bit-identical tables, loss_out and voxel gradients (plain, fused, fused + upstream);
  * exact plain gradients: bit for bit against ``exact_gather``, with no near-tie exclusions.
usage: python tests/fuzz_deterministic.py [cases] [seed]"""
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
import numpy as np
import torch

from spsg_b200 import _native as N
from spsg_b200 import synthetic as S
from tests import gather_oracle as O

SCHEDULES = (0, N.SPSG_FLAG_SMEM_MAPS, N.SPSG_FLAG_GLOBAL_MAPS, N.SPSG_FLAG_NO_BRICK_SKIP, N.SPSG_FLAG_NO_CLIP)
DIMS = S.DIMS_ZYX


def room(dev, B, seed=0, view_payload=0):
    """B chunks of the synthetic room with the voxel id in the normal payload: (N,3) rows (v + 1, 0.5, -0.25), or with
    view_payload = F per-view rows (v + 1, f + 0.5, -0.25) of an (N,F,3) payload."""
    batch = S.make_batch(list(range(seed, seed + B)))
    t = {k: torch.from_numpy(np.ascontiguousarray(batch[k])).to(dev) for k in ("locs", "sdf", "color", "semantic")}
    n = batch["locs"].shape[0]
    if view_payload:
        p = np.empty((n, view_payload, 3), np.float32)
        p[:, :, 0] = np.arange(1, n + 1, dtype=np.float32)[:, None]
        p[:, :, 1] = np.arange(view_payload, dtype=np.float32)[None, :] + 0.5
        p[:, :, 2] = -0.25
        t["normal"] = torch.from_numpy(p).to(dev)
    else:
        t["normal"] = torch.from_numpy(O.voxel_normals(n)).to(dev)
    return t, n, batch


def cameras(images, rng, w, h, close=1.0):
    """(I,4,4) camera->grid and (I,4) intrinsics; a fraction ``close`` of the cameras 15-25 voxels (0.3-0.5 m) in front of
    one of the room's two walls, above the sphere and the box, the others on the usual circle."""
    far, _ = S.make_views(images, 1, seed=int(rng.integers(1 << 30)))
    mats = []
    for i in range(images):
        if rng.random() >= close:
            mats.append(far[i])
            continue
        d, a, z = rng.uniform(15.0, 25.0), rng.uniform(15.0, 45.0), rng.uniform(55.0, 75.0)
        if rng.random() < 0.5:
            eye, tgt = (a, 56.7 - d, z), (a + rng.uniform(-6, 6), 62.0, z + rng.uniform(-8, 4))
        else:
            eye, tgt = (57.2 - d, a, z), (62.0, a + rng.uniform(-6, 6), z + rng.uniform(-8, 4))
        mats.append(S.look_at(eye, tgt))
    intr = np.tile(np.asarray(S.INTRINSICS, np.float32), (images, 1))
    intr[:, 0] *= w / S.WIDTH
    intr[:, 2] = (intr[:, 2] + 0.5) * w / S.WIDTH - 0.5
    intr[:, 1] *= h / S.HEIGHT
    intr[:, 3] = (intr[:, 3] + 0.5) * h / S.HEIGHT - 0.5
    return np.stack(mats).astype(np.float32), intr.astype(np.float32)


def raycaster(dev, B, F, w, h, n, max_pix, flags):
    from spsg_b200.raycast_rgbd import RaycastRGBD
    m = RaycastRGBD(B, DIMS, w, h, 0.0, 300.0, S.THRESH_SAMPLE_DIST, S.RAY_INCREMENT, max_num_frames=F,
                    max_num_locs_per_sample=n // B + 1, max_pixels_per_voxel=max_pix, device=dev)
    m.flags = flags
    return m


# ---- oracle ------------------------------------------------------------------------------------------------------------

def voxel_of_pixels(depth, normal):
    """(I, H*W) int64 voxel id from the renderings, -1 = miss (normal channel 0 carries v + 1)."""
    i = depth.shape[0]
    d = depth.reshape(i, -1)
    hit = d != -np.inf
    v = np.where(hit, normal.reshape(i, d.shape[1], 3)[..., 0], 0.0).astype(np.int64) - 1
    return np.where(hit, v, -1)


class Canonical:
    """The canonical tables of a rendering: entry ``rank`` of row ``row`` is pixel ``pix`` of image ``img``; ``cnt`` per row."""


def canonical_tables(vox, chunk, views, max_pix):
    n = chunk.shape[0]
    img, pix = np.nonzero(vox >= 0)
    v = vox[img, pix]
    assert bool((img // views == chunk[v]).all()), "a voxel was rendered into another chunk's image"
    row = (img % views) * n + v
    order = np.lexsort((pix, row))
    row, pix, img = row[order], pix[order], img[order]
    rank = np.arange(row.size) - np.searchsorted(row, row, side="left")
    keep = rank < max_pix
    c = Canonical()
    c.row, c.rank, c.pix, c.img = row[keep], rank[keep], pix[keep], img[keep]
    c.cnt = np.bincount(row, minlength=views * n)
    c.n, c.views, c.max_pix, c.P = n, views, max_pix, vox.shape[1]
    return c


def check_tables(c, mapping, num, what=""):
    """Counts equal |S(v, f)|, entries [0, min(cnt, P)) equal sorted(S(v, f))[:P].  Returns (rows hit, rows overflowed)."""
    num = num[:c.views * c.n].astype(np.int64)
    bad = np.nonzero(num != c.cnt)[0]
    assert bad.size == 0, "%s: %d counts differ from the renderings (row %d: %d vs %d)" % (
        what, bad.size, bad[0], num[bad[0]], c.cnt[bad[0]])
    got = mapping[c.row, c.rank]
    bad = np.nonzero(got != c.pix)[0]
    assert bad.size == 0, "%s: %d table entries are not the canonical ones (row %d slot %d: %d, want %d)" % (
        what, bad.size, c.row[bad[0]], c.rank[bad[0]], got[bad[0]], c.pix[bad[0]])
    return int((c.cnt > 0).sum()), int((c.cnt > c.max_pix).sum())


def exact_gather(c, G):
    """The plain backward over canonical tables, emulated operation by operation: per row a sequential float64 sum of the
    entries' fp32 rows in table order, times fl32(1/cnt) in double, rounded once to fp32; the views' means then added in
    view order in fp32 onto 0.  G: (num_pixels, 21) fp32 values in the kernel's channel order.  Returns (N, 21) fp32."""
    n, F = c.n, c.views
    Sm = np.zeros((F * n, 21))
    gpix = c.img * c.P + c.pix
    for r in range(c.max_pix):
        sel = c.rank == r
        Sm[c.row[sel]] += G[gpix[sel]]  # one entry per row per round: the rows of a round are distinct
    k = np.minimum(c.cnt, c.max_pix)
    live = k > 0
    inv = (1.0 / np.where(live, k, 1)).astype(np.float32).astype(np.float64)
    mean = (Sm * inv[:, None]).astype(np.float32)
    tot = np.zeros((n, 21), np.float32)
    for f in range(F):
        tot = np.where(live[f * n:(f + 1) * n, None], tot + mean[f * n:(f + 1) * n], tot)
    return tot


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.int32)


# ---- one run -----------------------------------------------------------------------------------------------------------

def targets(images, w, h, dev, rng):
    g = torch.Generator(device="cpu").manual_seed(int(rng.integers(1 << 30)))
    depth = torch.rand(images, h, w, generator=g) * 2.0 + 0.2
    depth[torch.rand(images, h, w, generator=g) < 0.05] = 0.0
    color = torch.rand(images, h, w, 3, generator=g)
    label = torch.randint(0, 15, (images, h, w), generator=g, dtype=torch.uint8)
    cw = torch.tensor(S.CLASS_WEIGHTS, dtype=torch.float32)
    return [x.to(dev) for x in (depth, color, label, cw)]


def run_once(m, t, view, intr, variant, seed, locs=None):
    """One forward + backward of raycaster m.  variant: 'plain' (autograd, random upstream images), 'fused', 'fused_up'
    (fused losses, plus upstream images of colour and normal).  Returns numpy (images, mapping, num, loss_out or None,
    grads (N, 21) fp32, upstream G or None)."""
    dev = view.device
    leaves = [t[k].clone().requires_grad_(True) for k in ("sdf", "color", "normal", "semantic")]
    locs = t["locs"] if locs is None else locs
    images = view.shape[0]
    rng = np.random.default_rng(seed)
    g = torch.Generator(device="cpu").manual_seed(seed)
    loss_out, G = None, None
    if variant == "plain":
        outs = m(locs, *leaves, view, intr)
        ups = [torch.randn(o.shape, generator=g).to(dev) for o in outs]
        torch.autograd.backward(outs, ups)
        gc, gd, gn, gs = (u.cpu().numpy() for u in ups)
        G = O.plain_pixel_grads(gc, gd, gn, gs)
        imgs = outs
    else:
        from spsg_b200.losses import render_with_2d_losses
        depth_t, color_t, label_t, cw = targets(images, m.width, m.height, dev, rng)
        total, terms, imgs = render_with_2d_losses(m, locs, *leaves, view, intr, images_depth=depth_t, images_color=color_t,
                                                   target2d_label=label_t, weight_semantic_class=cw,
                                                   voxelsize=S.VOXELSIZE, weight_color_loss=0.7, weight_semantic_loss=0.3,
                                                   differentiable_images=variant == "fused_up")
        obj = total
        if variant == "fused_up":
            finite = lambda x: torch.where(torch.isfinite(x), x, torch.zeros_like(x))
            obj = obj + 1e-3 * (finite(imgs[0]) * torch.randn(imgs[0].shape, generator=g).to(dev)).sum() + \
                1e-3 * (finite(imgs[2]) * torch.randn(imgs[2].shape, generator=g).to(dev)).sum()
        obj.backward()
        loss_out = torch.cat([terms, total[None]]).detach().cpu().numpy()
    torch.cuda.synchronize()
    d_sdf, d_col, d_nrm, d_sem = (x.grad for x in leaves)
    n = t["sdf"].shape[0]
    grads = np.concatenate([d_sem.reshape(n, 14).cpu().numpy(), d_col.reshape(n, 3).cpu().numpy(),
                            d_sdf.reshape(n, 1).cpu().numpy(), d_nrm.reshape(n, -1).cpu().numpy()], 1)
    im = [x.detach().cpu().numpy() for x in imgs]
    return im, m.mapping3dto2d.cpu().numpy(), m.mapping3dto2d_num.cpu().numpy(), loss_out, grads, G


def check_case(dev, B, F, max_pix, w, h, close, variant, seed, flags=0, per_view=False, what="", exact=True):
    """Tables against the renderings, schedule independence across SCHEDULES, and (plain, shared normals) exact gradients.
    Returns (rows hit, rows overflowed)."""
    t, n, batch = room(dev, B, seed, view_payload=F if per_view else 0)
    rng = np.random.default_rng(seed)
    view, intr = cameras(B * F, rng, w, h, close)
    view, intr = torch.from_numpy(view).to(dev), torch.from_numpy(intr).to(dev)
    chunk = batch["locs"][:, 3]
    ref = None
    stats = (0, 0)
    for sched in SCHEDULES:
        m = raycaster(dev, B, F, w, h, n, max_pix, N.SPSG_FLAG_DETERMINISTIC | flags | sched)
        im, mapping, num, loss_out, grads, G = run_once(m, t, view, intr, variant, seed)
        tag = "%s sched=%#x" % (what, sched)
        if ref is None:
            vox = voxel_of_pixels(im[1], im[2])
            c = canonical_tables(vox, chunk, F, max_pix)
            stats = check_tables(c, mapping, num, tag)
            if variant == "plain" and exact and not per_view:
                want = exact_gather(c, G)
                bad = bits(grads) != bits(want)
                assert not bad.any(), "%s: %d gradient entries differ from the exact emulation (first %s: %r vs %r)" % (
                    tag, int(bad.sum()), np.argwhere(bad)[0], grads[bad][0], want[bad][0])
            used = np.arange(max_pix)[None, :] < np.minimum(num[:F * n], max_pix)[:, None]
            ref = (im, np.where(used, mapping[:F * n], -1), num[:F * n], loss_out, grads)
            continue
        used = np.arange(max_pix)[None, :] < np.minimum(num[:F * n], max_pix)[:, None]
        for a, b in zip(im, ref[0]):
            assert np.array_equal(bits(a), bits(b)), "%s: renderings differ across schedules" % tag
        assert np.array_equal(num[:F * n], ref[2]), "%s: counts differ across schedules" % tag
        assert np.array_equal(np.where(used, mapping[:F * n], -1), ref[1]), "%s: tables differ across schedules" % tag
        if loss_out is not None:
            assert np.array_equal(bits(loss_out), bits(ref[3])), "%s: loss_out %r vs %r" % (tag, loss_out, ref[3])
        assert np.array_equal(bits(grads), bits(ref[4])), "%s: %d gradient entries differ across schedules" % (
            tag, int((bits(grads) != bits(ref[4])).sum()))
    return stats


def draw(rng):
    return dict(B=int(rng.integers(1, 9)), F=int(rng.integers(1, 6)), max_pix=int(rng.choice([1, 2, 7, 16, 33, 64])),
                wh=[(320, 256), (160, 128), (88, 60)][int(rng.integers(3))], close=float(rng.choice([1.0, 0.7, 0.3])),
                variant=str(rng.choice(["plain", "fused", "fused_up"])), per_view=bool(rng.random() < 0.2),
                flags=int(rng.choice([0, N.SPSG_FLAG_DETERMINISTIC_GRADS, N.SPSG_FLAG_RECORD_HITS])))


def run_case(c, dev, seed):
    w, h = c["wh"]
    B = c["B"] if w * h * c["B"] * c["F"] <= 12 * 320 * 256 else max(1, 12 * 320 * 256 // (w * h * c["F"]))
    return check_case(dev, B, c["F"], c["max_pix"], w, h, c["close"], c["variant"], seed, flags=c["flags"],
                      per_view=c["per_view"] and c["F"] > 1, what="case %s seed %d" % (c, seed))


def run(cases=100, seed0=0, dev=None):
    """Returns the number of failing cases."""
    dev = dev or torch.device("cuda", 0)
    fails, hit, over = 0, 0, 0
    t0 = time.time()
    for k in range(cases):
        rng = np.random.default_rng(seed0 * 100003 + k)
        c = draw(rng)
        try:
            h, o = run_case(c, dev, seed0 * 100003 + k)
            hit += h
            over += o
        except AssertionError as e:
            fails += 1
            print("MISMATCH:", e, flush=True)
    print("deterministic fuzz: %d cases, %d mismatching, %d (voxel, view) rows hit, %d overflowed (%.0f s)"
          % (cases, fails, hit, over, time.time() - t0), flush=True)
    return fails


if __name__ == "__main__":
    sys.exit(1 if run(int(sys.argv[1]) if len(sys.argv) > 1 else 100, int(sys.argv[2]) if len(sys.argv) > 2 else 0) else 0)
