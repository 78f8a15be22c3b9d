"""Randomised sweep of the all-pixels mode (SPSG_FLAG_ALL_PIXELS, ``RaycastRGBD(..., max_pixels_per_voxel=None)``);
tests/test_gpu_all_pixels.py runs a seeded slice under pytest and uses the same helpers.

Each case renders random chunks of the synthetic room (B = 1-8, F = 1-3) from random cameras -- close ones (0.3-0.5 m from a
wall, where most (voxel, view) rows get more than 64 pixels), some of them zoomed so that single rows cover thousands of
pixels, mixed with far ones -- and checks, with the voxel id in the normal payload so that every pixel's voxel is known from
the renderings:
  * counts: mapping3dto2d_num equals |S(v, f)|, the number of pixels of view f whose voxel is v;
  * with SPSG_FLAG_DETERMINISTIC, plain variant: the voxel gradients equal, bit for bit, the emulation of a gather over ALL
    of S(v, f) in ascending pixel order (per-view normal rows too);
  * fused and fused + upstream variants: the gradients against the float64 gather of the recomputed pixel gradients, at the
    bars of tests/gather_oracle.py;
  * schedule independence: renderings, counts, loss_out and gradients bit-identical across the schedule flags.
usage: python tests/fuzz_all_pixels.py [cases] [seed]"""
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
from tests import fuzz_deterministic as D
from tests import gather_oracle as O

SCHEDULES = D.SCHEDULES
ALL = N.SPSG_FLAG_ALL_PIXELS
DET = N.SPSG_FLAG_DETERMINISTIC
SMEM_SORT = 4096  # kSegSmemSort of spsg_segments.cuh: longer rows are rebuilt by the ordered compaction


def cameras(images, rng, w, h, close, zoom=1.0):
    """fuzz_deterministic.cameras with the focal lengths multiplied by ``zoom`` (larger: fewer voxels, more pixels each)."""
    view, intr = D.cameras(images, rng, w, h, close)
    intr[:, 0] *= zoom
    intr[:, 1] *= zoom
    return view, intr


def all_tables(vox, chunk, views):
    """``canonical_tables`` with no cap: max_pix = the largest row (every rank of every row kept)."""
    c = D.canonical_tables(vox, chunk, views, vox.shape[1])
    c.max_pix = max(int(c.cnt.max()), 1)
    return c


def exact_gather(c, G):
    """fuzz_deterministic.exact_gather, with each rank's entries taken from one sorted slice instead of a mask over all
    entries (the loop runs to the longest row, thousands of ranks here).  Returns (tot (N, 21) fp32 summed over views in
    view order, mean (F*N, 21) fp32 per row, live (F*N,) rows that received pixels)."""
    n, F = c.n, c.views
    Sm = np.zeros((F * n, 21))
    gpix = c.img * c.P + c.pix
    order = np.argsort(c.rank, kind="stable")
    rank = c.rank[order]
    bounds = np.searchsorted(rank, np.arange(int(rank.max()) + 2 if rank.size else 1))
    for r in range(bounds.size - 1):
        sel = order[bounds[r]:bounds[r + 1]]
        Sm[c.row[sel]] += G[gpix[sel]]  # one entry per row per rank: the rows of a rank are distinct
    k = np.minimum(c.cnt, c.max_pix)
    live = k > 0
    inv = (1.0 / np.where(live, k, 1)).astype(np.float32).astype(np.float64)
    mean = (Sm * inv[:, None]).astype(np.float32)
    tot = np.zeros((n, 21), np.float32)
    for f in range(F):
        tot = np.where(live[f * n:(f + 1) * n, None], tot + mean[f * n:(f + 1) * n], tot)
    return tot, mean, live


def expected_exact(c, G, per_view):
    """The deterministic plain gradients as run_once returns them: (N, 21), or (N, 18 + 3F) with per-view normal rows."""
    tot, mean, live = exact_gather(c, G)
    if not per_view:
        return tot
    rows = np.where(live[:, None], mean[:, 18:21], np.float32(0)).reshape(c.views, c.n, 3).transpose(1, 0, 2)
    return np.concatenate([tot[:, :18], rows.reshape(c.n, 3 * c.views)], 1)


def fused_expectation(c, im, seed, variant):
    """(gather_oracle.Gather, tables) of the fused variants of run_once: the same seeded targets and upstream images."""
    images, h, w = im[1].shape
    depth_t, color_t, label_t, cw = (x.cpu().numpy() for x in D.targets(images, w, h, torch.device("cpu"),
                                                                        np.random.default_rng(seed)))
    up = None
    if variant == "fused_up":
        g = torch.Generator(device="cpu").manual_seed(seed)
        k = np.float32(1e-3)
        uc = torch.randn(im[0].shape, generator=g).numpy() * k
        un = torch.randn(im[2].shape, generator=g).numpy() * k
        up = (np.where(np.isfinite(im[0]), uc, 0).astype(np.float32), None,
              np.where(np.isfinite(im[2]), un, 0).astype(np.float32), None)
    G, mag, bound, _ = O.fused_pixel_grads(im[0], im[1], im[3], target_depth=depth_t, target_color=color_t, label=label_t,
                                           class_weight=cw, voxelsize=S.VOXELSIZE, weights=(1.0, 0.7, 0.3), upstream=up)
    return O.gather(tables(c), G, pixel_bound=bound, mag=mag)


def tables(c):
    """The uncapped tables as gather_oracle's validated pixel sets."""
    return O.Tables(c.n, c.views, c.row, c.img * c.P + c.pix, c.cnt, np.zeros(0, np.int64))


def check_case(dev, B, F, w, h, close, variant, seed, flags=0, per_view=False, zoom=1.0, schedules=SCHEDULES, what=""):
    """Counts, exact (deterministic plain) or bounded (fused) gradients, and schedule independence across ``schedules``.
    Returns (rows hit, rows over 64, largest row)."""
    t, n, batch = D.room(dev, B, seed, view_payload=F if per_view else 0)
    view, intr = cameras(B * F, np.random.default_rng(seed), w, h, close, zoom)
    view, intr = torch.from_numpy(view).to(dev), torch.from_numpy(intr).to(dev)
    chunk = batch["locs"][:, 3]
    ref, stats = None, (0, 0, 0)
    for sched in schedules:
        m = D.raycaster(dev, B, F, w, h, n, None, ALL | flags | sched)
        assert m.mapping3dto2d.numel() == 0
        im, _, num, loss_out, grads, G = D.run_once(m, t, view, intr, variant, seed)
        tag = "%s sched=%#x" % (what, sched)
        num = num[:F * n]
        if ref is None:
            c = all_tables(D.voxel_of_pixels(im[1], im[2]), chunk, F)
            bad = np.nonzero(num != c.cnt)[0]
            assert bad.size == 0, "%s: %d counts differ from the renderings (row %d: %d vs %d)" % (
                tag, bad.size, bad[0], num[bad[0]], c.cnt[bad[0]])
            if variant == "plain" and flags & DET:
                want = expected_exact(c, G, per_view)
                bad = D.bits(grads) != D.bits(want)
                assert not bad.any(), "%s: %d gradient entries differ from the exact emulation (first %s: %r vs %r)" % (
                    tag, int(bad.sum()), np.argwhere(bad)[0], grads[bad][0], want[bad][0])
            elif variant == "plain" and not per_view:
                O.compare(grads, O.gather(tables(c), G), tag)
            elif not per_view:
                O.compare(grads, fused_expectation(c, im, seed, variant), tag)
            stats = (int((c.cnt > 0).sum()), int((c.cnt > 64).sum()), int(c.cnt.max()))
            ref = (im, num, loss_out, grads)
            continue
        for a, b in zip(im, ref[0]):
            assert np.array_equal(D.bits(a), D.bits(b)), "%s: renderings differ across schedules" % tag
        assert np.array_equal(num, ref[1]), "%s: counts differ across schedules" % tag
        if loss_out is not None:
            assert np.array_equal(D.bits(loss_out), D.bits(ref[2])), "%s: loss_out %r vs %r" % (tag, loss_out, ref[2])
        assert np.array_equal(D.bits(grads), D.bits(ref[3])), "%s: %d gradient entries differ across schedules" % (
            tag, int((D.bits(grads) != D.bits(ref[3])).sum()))
    return stats


def draw(rng):
    return dict(B=int(rng.integers(1, 9)), F=int(rng.integers(1, 4)),
                wh=[(320, 256), (160, 128), (88, 60)][int(rng.integers(3))], close=float(rng.choice([1.0, 0.7, 0.3])),
                zoom=float(rng.choice([1.0, 1.0, 2.0, 4.0])), variant=str(rng.choice(["plain", "fused", "fused_up"])),
                per_view=bool(rng.random() < 0.25), det=bool(rng.random() < 0.75),
                flags=int(rng.choice([0, N.SPSG_FLAG_DETERMINISTIC_GRADS, N.SPSG_FLAG_RECORD_HITS])))


def run_case(c, dev, seed):
    w, h = c["wh"]
    B = c["B"] if w * h * c["B"] * c["F"] <= 8 * 320 * 256 else max(1, 8 * 320 * 256 // (w * h * c["F"]))
    # deterministic: two schedules (the default and one drawn) bit-identical; default mode: one run, bounded check only
    sched = (0, SCHEDULES[1 + seed % 4]) if c["det"] else (0,)
    return check_case(dev, B, c["F"], w, h, c["close"], c["variant"], seed, flags=c["flags"] | (DET if c["det"] else 0),
                      per_view=c["per_view"] and c["F"] > 1, zoom=c["zoom"], schedules=sched,
                      what="case %s seed %d" % (c, seed))


def run(cases=100, seed0=0, dev=None):
    """Returns the number of failing cases."""
    dev = dev or torch.device("cuda", 0)
    fails, hit, over, longest = 0, 0, 0, 0
    t0 = time.time()
    for k in range(cases):
        rng = np.random.default_rng(seed0 * 100003 + k)
        c = draw(rng)
        try:
            h, o, mx = run_case(c, dev, seed0 * 100003 + k)
            hit += h
            over += o
            longest = max(longest, mx)
        except AssertionError as e:
            fails += 1
            print("MISMATCH:", e, flush=True)
    print("all-pixels fuzz: %d cases, %d mismatching, %d (voxel, view) rows hit, %d over 64 pixels, largest row %d pixels "
          "(%.0f s)" % (cases, fails, hit, over, longest, time.time() - t0), flush=True)
    return fails


if __name__ == "__main__":
    sys.exit(1 if run(int(sys.argv[1]) if len(sys.argv) > 1 else 100, int(sys.argv[2]) if len(sys.argv) > 2 else 0) else 0)
