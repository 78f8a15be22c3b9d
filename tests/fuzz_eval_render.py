"""Helpers and a random sweep for the eval render (``losses.evaluate_2d``, spsg_raycast_eval; tests/test_gpu_eval_render.py).

    python -m tests.fuzz_eval_render [cases] [seed]

The eval render marches exactly like the fused forward and forms each warp's six loss partials with the same per-pixel
arithmetic, so on the same voxels, cameras and targets ``evaluate_2d`` must give:
  * the normalisers loss_out[4:7] of ``fused_forward`` bit for bit, and its terms and total within 1e-6 relative (only the
    double summation order differs);
  * ``labels_from_render`` of the forward's semantic image, bit for bit, as its label map;
  * ``bincount(min(target, C) * (C + 1) + labels)`` as its confusion matrix, exactly.
Every case draws C in 1..64, B chunks, F views, an image size, a grid (the 128x64x64 chunk or one whose maps do not fit in
shared memory), a ray increment, a scene, cameras, empty chunks, targets (each term on or off, colour weights, class
weights, labels at and above C), a debug flag and an index route (int64 rows, packed rows, prebuilt index).
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))  # run as a script from anywhere

import numpy as np
import torch

from spsg_b200 import _native as N
from spsg_b200 import losses
from spsg_b200 import raycast_rgbd_cuda as rc
from spsg_b200 import sparsify
from spsg_b200 import synthetic as S
from tests import fuzz_label_render as L

BIG_DIMS = L.BIG_DIMS
DEBUG_FLAGS = L.DEBUG_FLAGS
TERMS_ALL = ("depth", "color", "semantic")


def payload(n, C, seed, dev):
    g = torch.Generator(device="cpu").manual_seed(seed)
    color = torch.rand(n, 3, generator=g)
    logits = torch.randn(n, C, generator=g) * 2.0
    return color.contiguous().to(dev), logits.contiguous().to(dev)


def targets(images, h, w, C, seed, dev, terms=TERMS_ALL, weight_color=True, class_weight=True):
    """(images_depth, images_color, weight_color, target2d_label, class_weight): depth with holes, labels 0..C + 3 (some
    at and above C), any of them None where switched off."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    depth = torch.rand(images, h, w, generator=g) * 3.0
    depth[torch.rand(images, h, w, generator=g) < 0.1] = 0.0
    color = torch.rand(images, h, w, 3, generator=g)
    wc = torch.rand(images, h, w, generator=g) + 0.5
    lab = torch.randint(0, C + 4, (images, h, w), generator=g).to(torch.uint8)
    cw = torch.rand(C, generator=g) * 1.5 + 0.25
    put = lambda t, on: t.contiguous().to(dev) if on else None  # noqa: E731
    return (put(depth, "depth" in terms), put(color, "color" in terms), put(wc, "color" in terms and weight_color),
            put(lab, "semantic" in terms), put(cw, "semantic" in terms and class_weight))


def reference(m, locs, sdf, color, logits, view, intr, tg, voxelsize=0.02, weights=(1.0, 0.7, 0.3)):
    """The fused forward on the same inputs: (loss_out, label map, confusion or None, renderings)."""
    C = m.num_classes
    normals = torch.zeros(locs.shape[0], 3, device=sdf.device)
    with torch.no_grad():
        _, _, out = losses.fused_forward(m, locs, sdf, color, normals, logits, view, intr,
                                         tg + (voxelsize, weights), False)
    images = view.shape[0]
    sem = m.image_semantic[:images]
    lab = losses.labels_from_render(sem)
    conf = None
    if tg[3] is not None:
        conf = torch.bincount(tg[3].long().clamp(max=C).flatten() * (C + 1) + lab.long().flatten(),
                              minlength=(C + 1) ** 2).view(C + 1, C + 1)
    torch.cuda.synchronize()
    imgs = tuple(x[:images].clone() for x in (m.image_color, m.image_depth, m.image_semantic))
    return out.clone(), lab.clone(), conf, imgs


def evaluate(m, locs, sdf, color, logits, view, intr, tg, voxelsize=0.02, weights=(1.0, 0.7, 0.3), labels=True):
    total, terms, conf, lab = losses.evaluate_2d(
        m, locs, sdf, color, logits, view, intr, images_depth=tg[0], images_color=tg[1], weight_color=tg[2],
        target2d_label=tg[3], weight_semantic_class=tg[4], voxelsize=voxelsize, weight_depth_loss=weights[0],
        weight_color_loss=weights[1], weight_semantic_loss=weights[2], labels=labels)
    torch.cuda.synchronize()
    return total, terms, conf, lab


def loss_block(total, terms):
    """loss_out[0:8] of an evaluate_2d result (total and terms are views of it)."""
    return terms.as_strided((N.SPSG_LOSS_OUT_FLOATS,), (1,))


def compare(got, want, what):
    total, terms, conf, lab = got
    out, wl, wc, _ = want
    block = loss_block(total, terms)
    assert torch.equal(block[4:7].view(torch.int32), out[4:7].view(torch.int32)), \
        "%s: normalisers %s vs %s" % (what, block[4:7].tolist(), out[4:7].tolist())
    a, b = block[:4].double(), out[:4].double()
    same = (a == b) | (torch.isnan(a) & torch.isnan(b)) | ((a - b).abs() <= 1e-6 * b.abs())
    assert bool(same.all()), "%s: terms %s vs %s" % (what, a.tolist(), b.tolist())
    if lab is not None:
        bad = int((lab != wl).sum())
        assert bad == 0, "%s: %d of %d label pixels differ" % (what, bad, lab.numel())
    assert (conf is None) == (wc is None), what
    if conf is not None:
        assert torch.equal(conf, wc), "%s: confusion matrices differ in %d cells" % (what, int((conf != wc).sum()))


def permuted(m, locs, sdf, B, dims):
    """Rows of sparsify_predictions(..., raycaster=m) over a dense SDF head holding exactly these voxels (the prebuilt index
    route), and for each of its rows the index of the caller's row."""
    outside = torch.full((B, 1) + tuple(dims), 10.0, device=locs.device)
    outside[locs[:, 3], 0, locs[:, 0], locs[:, 1], locs[:, 2]] = sdf[:, 0]
    plocs, psdf = sparsify.sparsify_predictions(outside.contiguous(), S.TRUNCATION, raycaster=m)
    idx = torch.full((B,) + tuple(dims), -1, dtype=torch.int64, device=locs.device)
    idx[locs[:, 3], locs[:, 0], locs[:, 1], locs[:, 2]] = torch.arange(locs.shape[0], device=locs.device)
    return plocs, psdf, idx[plocs[:, 3], plocs[:, 0], plocs[:, 1], plocs[:, 2]]


def check_case(dev, C, B, F, w, h, seed, dims=S.DIMS_ZYX, kind="room", inc=S.RAY_INCREMENT, flags=0, route="int64",
               empty=(), close=0.3, away=0.0, n_zero=False, terms=TERMS_ALL, weight_color=True, class_weight=True,
               generic=False):
    """evaluate_2d against the fused forward on the same voxels, cameras and targets.  Returns the number of pixels hit."""
    rng = np.random.default_rng(seed)
    locs, sdf = L.scene(dev, B, dims, seed, kind)
    locs, sdf = L.drop_chunks(locs, sdf, empty)
    if n_zero:
        locs, sdf = locs[:0].contiguous(), sdf[:0].contiguous()
    n = locs.shape[0]
    color, logits = payload(n, C, seed + 1, dev)
    view, intr = L.cameras(dev, B * F, rng, w, h, dims, close, away)
    tg = targets(B * F, h, w, C, seed + 2, dev, terms, weight_color, class_weight)
    ref = L.module(dev, B, F, w, h, n, C, dims, inc, flags | (N.SPSG_FLAG_GENERIC_SEMANTIC if generic else 0))
    want = reference(ref, locs, sdf, color, logits, view, intr, tg)
    m = L.module(dev, B, F, w, h, n, C, dims, inc, flags)
    if route == "packed":
        got = evaluate(m, rc.pack_locs_host(locs.cpu(), B, dims).to(dev), sdf, color, logits, view, intr, tg)
    elif route == "prebuilt":
        plocs, psdf, perm = permuted(m, locs, sdf, B, dims)
        seen = []
        real = N.lib.spsg_raycast_eval

        def spy(p, *args):
            seen.append(p._obj.flags)
            return real(p, *args)
        N.lib.spsg_raycast_eval = spy
        try:
            got = evaluate(m, plocs, psdf, color[perm].contiguous(), logits[perm].contiguous(), view, intr, tg)
        finally:
            N.lib.spsg_raycast_eval = real
        assert plocs.shape[0] == 0 or seen[0] & N.SPSG_FLAG_INDEX_PREBUILT, "the eval render did not take the prebuilt index"
    else:
        got = evaluate(m, locs, sdf, color, logits, view, intr, tg)
    compare(got, want, "C=%d B=%d F=%d %dx%d dims=%s %s inc=%g flags=%#x %s empty=%s terms=%s" % (
        C, B, F, w, h, tuple(dims), kind, inc, flags, route, tuple(empty), terms))
    return int((want[1] < C).sum())


def case(rng):
    c = L.case(rng)
    del c["n_zero"]
    terms = tuple(t for t in TERMS_ALL if rng.random() < 0.8)
    return dict(c, n_zero=bool(rng.random() < 0.03), terms=terms, weight_color=bool(rng.random() < 0.5),
                class_weight=bool(rng.random() < 0.5))


def run_case(dev, c):
    check_case(dev, c["C"], c["B"], c["F"], c["w"], c["h"], c["seed"], dims=c["dims"], kind=c["kind"], inc=c["inc"],
               flags=c["flags"], route=c["route"], empty=c["empty"], close=c["close"], away=c["away"], n_zero=c["n_zero"],
               terms=c["terms"], weight_color=c["weight_color"], class_weight=c["class_weight"])


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
    print("eval-render sweep: %d cases, %d mismatches" % (cases, len(fails)))
    for f in fails:
        print(f)
    sys.exit(1 if fails else 0)
