"""Helpers and a random sweep for the configurable semantic class count (tests/test_gpu_semantic_classes.py).

    python -m tests.fuzz_semantic_classes [cases] [seed]

Every case draws C in 1..64, B chunks, F views, an image size, cameras (far, or 0.3-0.5 m from a wall), extra flags and a
route (plain / fused / fused + upstream), and checks
  * geometry: colour, depth, normal renderings and mapping3dto2d_num bit-identical to the 14-class render of the same voxels
    (and, deterministic, the tables); every semantic pixel its hit voxel's payload row, misses -inf;
  * plain route, deterministic: the C-channel gradients bit-identical to 14-channel backwards of 14-channel windows;
  * fused routes: loss terms and voxel gradients against the literal PyTorch losses through the plain raycast.
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

DET, ALL = N.SPSG_FLAG_DETERMINISTIC, N.SPSG_FLAG_ALL_PIXELS
NINF = -float("inf")


def bits(t):
    return t.detach().contiguous().view(torch.int32)


def setup(dev, B, F, w, h, seed, close=0.5, per_view=False):
    t, n, batch = D.room(dev, B, seed, view_payload=F if per_view else 0)
    view, intr = D.cameras(B * F, np.random.default_rng(seed), w, h, close)
    return t, n, batch, torch.from_numpy(view).to(dev), torch.from_numpy(intr).to(dev)


def module(dev, B, F, w, h, n, C, flags):
    m = RaycastRGBD(B, S.DIMS_ZYX, w, h, S.DEPTH_MIN, S.DEPTH_MAX, S.THRESH_SAMPLE_DIST, S.RAY_INCREMENT,
                    max_num_frames=F, max_num_locs_per_sample=max(-(-n // B), 1),
                    max_pixels_per_voxel=None if flags & ALL else 64, device=dev, num_classes=C)
    m.flags |= flags & ~ALL
    return m


def logits(n, C, seed, dev):
    g = torch.Generator(device=dev).manual_seed(seed)
    return torch.randn(n, C, device=dev, generator=g) * 2.0


def _table(m, n, F):
    """(rows, P) registration table with the undefined entries (beyond num) set to -2; None without a table."""
    if m.mapping3dto2d.numel() == 0:
        return None
    num = m.mapping3dto2d_num[:n * F]
    tab = m.mapping3dto2d[:n * F]
    keep = torch.arange(tab.shape[1], device=tab.device)[None, :] < num[:, None]
    return torch.where(keep, tab, torch.full_like(tab, -2))


def render(dev, t, n, view, intr, B, F, w, h, C, flags, sem, locs=None):
    m = module(dev, B, F, w, h, n, C, flags)
    out = m(t["locs"] if locs is None else locs, t["sdf"], t["color"], t["normal"], sem, view, intr)
    torch.cuda.synchronize()
    return m, [o.clone() for o in out]


def check_render(dev, C, B, F, w, h, seed, flags=DET, close=0.5):
    t, n, batch, view, intr = setup(dev, B, F, w, h, seed, close)
    sem = logits(n, C, seed, dev)
    m, (col, dep, nrm, img) = render(dev, t, n, view, intr, B, F, w, h, C, flags, sem)
    m14, (col14, dep14, nrm14, _) = render(dev, t, n, view, intr, B, F, w, h, 14, flags, logits(n, 14, seed + 1, dev))
    for a, b, what in ((col, col14, "colour"), (dep, dep14, "depth"), (nrm, nrm14, "normal"),
                       (m.mapping3dto2d_num[:n * F], m14.mapping3dto2d_num[:n * F], "num")):
        assert torch.equal(bits(a), bits(b)), "C=%d: %s differs from the 14-class render" % (C, what)
    if flags & DET and not flags & ALL:
        assert torch.equal(_table(m, n, F), _table(m14, n, F)), "C=%d: tables differ" % C
    hit = dep != NINF
    vox = (nrm[..., 0] - 1).long()
    assert img.shape[-1] == C
    assert torch.equal(bits(img[hit]), bits(sem[vox[hit]])), "C=%d: a semantic pixel is not its voxel's row" % C
    assert bool((img[~hit] == NINF).all()), "C=%d: a miss is not -inf" % C
    return int(hit.sum())


def upstream_images(m, seed):
    g = torch.Generator(device=m.image_depth.device).manual_seed(seed)
    return [torch.randn(x.shape, device=x.device, generator=g) for x in (m.image_color, m.image_depth, m.image_normal,
                                                                           m.image_semantic)]


def _leaves(t, sem):
    return [x.clone().requires_grad_(True) for x in (t["sdf"], t["color"], t["normal"], sem)]


def plain_grads(dev, t, n, view, intr, B, F, w, h, C, flags, sem, gimg, locs=None):
    m = module(dev, B, F, w, h, n, C, flags)
    leaves = _leaves(t, sem)
    out = m(t["locs"] if locs is None else locs, *leaves, view, intr)
    grads = torch.autograd.grad(out, leaves, [g[:o.shape[0]] for g, o in zip(gimg, out)])
    torch.cuda.synchronize()
    return [g.clone() for g in grads]


def check_plain_grads(dev, C, B, F, w, h, seed, flags=DET, close=0.5):
    """C-channel plain backward against 14-channel backwards of the same images cut into windows of 14 channels: bit for
    bit with SPSG_FLAG_DETERMINISTIC; in the default mode (double sums rounded once, several views added with float
    atomics) within 1e-5, on cameras that overflow no table row unless the rows are uncapped (ALL_PIXELS)."""
    exact = bool(flags & DET)

    def same(a, b, what):
        if exact:
            assert torch.equal(bits(a), bits(b)), what
        else:
            assert torch.allclose(a, b, rtol=1e-5, atol=1e-6), what
    t, n, batch, view, intr = setup(dev, B, F, w, h, seed, close)
    sem = logits(n, C, seed, dev)
    gimg = upstream_images(module(dev, B, F, w, h, n, C, flags), seed + 1)
    got = plain_grads(dev, t, n, view, intr, B, F, w, h, C, flags, sem, gimg)
    for s in range(0, C, 14):
        k = min(14, C - s)
        pad = lambda x: torch.cat([x[..., s:s + k], torch.zeros(x.shape[:-1] + (14 - k,), device=dev)], -1).contiguous()
        want = plain_grads(dev, t, n, view, intr, B, F, w, h, 14, flags, pad(sem), gimg[:3] + [pad(gimg[3])])
        same(got[3][:, s:s + k], want[3][:, :k], "C=%d: semantic gradient window %d" % (C, s))
        if s == 0:
            for i, what in enumerate(("sdf", "colour", "normal")):
                same(got[i], want[i], "C=%d: %s gradient" % (C, what))


def targets(dev, B, F, w, h, C, seed, weights, ignore):
    g = torch.Generator(device=dev).manual_seed(seed + 99)
    I = B * F
    td = torch.rand(I, h, w, device=dev, generator=g) * 3.0
    td[torch.rand(I, h, w, device=dev, generator=g) < 0.2] = 0.0
    tc = torch.rand(I, h, w, 3, device=dev, generator=g)
    lab = torch.randint(0, C, (I, h, w), device=dev, generator=g)
    lab[torch.rand(I, h, w, device=dev, generator=g) < ignore] = C
    cw = torch.rand(C, device=dev, generator=g) + 0.5 if weights else None
    return td, tc, lab.to(torch.uint8), cw


def literal_losses(col, dep, sem, td, tc, lab, cw, vs, terms):
    """train.py:635-638, loss.py:246-257, train.py:744-746 with C logits (valid = label < C & logit0 != -inf)."""
    C = sem.shape[-1]
    vd = (dep != NINF) & (td != 0)
    ld = torch.mean(torch.abs(dep[vd] * vs - td[vd]))
    vc = col != NINF
    lc = torch.mean(torch.abs(col[vc] - tc[vc]))
    vsm = (lab < C) & (sem[..., 0] != NINF)
    ls = Fn.cross_entropy(sem[vsm].view(-1, C), lab[vsm].long(), weight=cw)
    return terms[0] * ld + terms[1] * lc + terms[2] * ls, torch.stack([ld, lc, ls])


def _close(got, want, tol, what):
    err = float((got - want).norm())
    scale = float(want.norm())
    assert err <= tol * scale + 1e-7, "%s: |err| %.3g vs |ref| %.3g" % (what, err, scale)


def check_losses(dev, C, B, F, w, h, seed, weights, ignore, terms, flags=DET, upstream=False, close=0.5):
    """(Deterministic tables by default: both sides then average an overflowing row over the same pixels.)"""
    vs = 0.02
    t, n, batch, view, intr = setup(dev, B, F, w, h, seed, close)
    sem = logits(n, C, seed, dev)
    td, tc, lab, cw = targets(dev, B, F, w, h, C, seed, weights, ignore)
    # fused
    m = module(dev, B, F, w, h, n, C, flags)
    leaves = _leaves(t, sem)
    total, t3, imgs = losses.render_with_2d_losses(m, t["locs"], *leaves, view, intr, images_depth=td, images_color=tc,
                                                   target2d_label=lab, weight_semantic_class=cw, voxelsize=vs,
                                                   weight_depth_loss=terms[0], weight_color_loss=terms[1],
                                                   weight_semantic_loss=terms[2], differentiable_images=upstream)
    gimg = upstream_images(m, seed + 5) if upstream else None
    obj = total
    if upstream:
        obj = obj + sum((torch.where(torch.isfinite(x), x, torch.zeros_like(x)) * g).sum() for x, g in zip(imgs, gimg))
    got = torch.autograd.grad(obj, leaves)
    got_terms = t3.clone()
    # literal losses through the plain raycast
    m2 = module(dev, B, F, w, h, n, C, flags)
    leaves2 = _leaves(t, sem)
    col, dep, nrm, img = m2(t["locs"], *leaves2, view, intr)
    ref_total, ref_terms = literal_losses(col, dep, img, td, tc, lab, cw, vs, terms)
    obj2 = ref_total
    if upstream:
        obj2 = obj2 + sum((torch.where(torch.isfinite(x), x, torch.zeros_like(x)) * g).sum()
                          for x, g in zip((col, dep, nrm, img), gimg))
    want = torch.autograd.grad(obj2, leaves2)
    assert torch.allclose(got_terms, ref_terms.detach(), rtol=1e-5, atol=1e-6), (C, got_terms, ref_terms)
    assert torch.allclose(total.detach(), ref_total.detach(), rtol=1e-5, atol=1e-6), (C, total, ref_total)
    for g, r, what in zip(got, want, ("sdf", "colour", "normal", "semantic")):
        _close(g, r, 1e-3, "C=%d %s gradient" % (C, what))
    # stand-alone losses on the renderings
    ci, di, si = (x.detach().clone().requires_grad_(True) for x in (col, dep, img))
    tot_s, terms_s = losses.losses_2d(ci, di, si, td, tc, None, lab, cw, vs, *terms)
    gs = torch.autograd.grad(tot_s, (ci, di, si))
    cj, dj, sj = (x.detach().clone().requires_grad_(True) for x in (col, dep, img))
    tot_l, terms_l = literal_losses(cj, dj, sj, td, tc, lab, cw, vs, terms)
    gl = torch.autograd.grad(tot_l, (cj, dj, sj))
    assert torch.allclose(terms_s, terms_l.detach(), rtol=1e-5, atol=1e-6), (C, terms_s, terms_l)
    for g, r, what in zip(gs, gl, ("colour", "depth", "semantic")):
        _close(g, r, 1e-3, "C=%d stand-alone %s gradient" % (C, what))


ROUTE_KEYS = ("color", "depth", "normal", "semantic", "num", "table")


def run_all_routes(dev, C, B, F, w, h, seed, flags, per_view=False, close=1.0):
    """Renderings, tables, loss_out and the gradients of the plain, fused and fused + upstream routes of one
    configuration, keyed by name."""
    t, n, batch, view, intr = setup(dev, B, F, w, h, seed, close, per_view)
    sem = logits(n, C, seed, dev)
    res = {}
    m = module(dev, B, F, w, h, n, C, flags)
    gimg = upstream_images(m, seed + 1)
    leaves = _leaves(t, sem)
    out = m(t["locs"], *leaves, view, intr)
    for k, o in zip(ROUTE_KEYS, out):
        res[k] = o.detach().clone()
    res["num"] = m.mapping3dto2d_num[:n * F].clone()
    tab = _table(m, n, F)
    if tab is not None and flags & DET:
        res["table"] = tab
    for k, g in zip(("sdf", "colour", "normal", "semantic"), torch.autograd.grad(out, leaves, gimg)):
        res["grad_plain_" + k] = g.clone()
    td, tc, lab, cw = targets(dev, B, F, w, h, C, seed, True, 0.2)
    for up in (False, True):
        m = module(dev, B, F, w, h, n, C, flags)
        leaves = _leaves(t, sem)
        total, t3, imgs = losses.render_with_2d_losses(m, t["locs"], *leaves, view, intr, images_depth=td, images_color=tc,
                                                       target2d_label=lab, weight_semantic_class=cw,
                                                       differentiable_images=up)
        obj = total
        if up:
            obj = obj + sum((torch.where(torch.isfinite(x), x, torch.zeros_like(x)) * g).sum() for x, g in zip(imgs, gimg))
        tag = "fused_up" if up else "fused"
        for k, g in zip(("sdf", "colour", "normal", "semantic"), torch.autograd.grad(obj, leaves)):
            res["grad_%s_%s" % (tag, k)] = g.clone()
        res["loss_%s" % tag] = torch.cat([total.detach().view(1), t3.detach()])
    torch.cuda.synchronize()
    return res


def check_routes(dev, C):
    """Packed locs render and differentiate like int64 locs; retain_graph gives twice the gradient."""
    B, F, w, h = 2, 1, 160, 128
    t, n, batch, view, intr = setup(dev, B, F, w, h, 17)
    sem = logits(n, C, 17, dev)
    packed = rc.pack_locs_host(t["locs"].cpu(), B, S.DIMS_ZYX).to(dev)
    gimg = upstream_images(module(dev, B, F, w, h, n, C, DET), 3)
    a = plain_grads(dev, t, n, view, intr, B, F, w, h, C, DET, sem, gimg)
    b = plain_grads(dev, t, n, view, intr, B, F, w, h, C, DET, sem, gimg, locs=packed)
    for x, y in zip(a, b):
        assert torch.equal(bits(x), bits(y))
    m = module(dev, B, F, w, h, n, C, DET)
    leaves = _leaves(t, sem)
    out = m(t["locs"], *leaves, view, intr)
    obj = sum((torch.where(torch.isfinite(x), x, torch.zeros_like(x)) * g).sum() for x, g in zip(out, gimg))
    obj.backward(retain_graph=True)
    first = [x.grad.clone() for x in leaves]
    obj.backward()
    for x, g1 in zip(leaves, first):
        assert torch.equal(bits(x.grad), bits(g1 * 2))
    assert torch.equal(bits(first[3]), bits(a[3]))


def case(rng):
    C = int(rng.integers(1, 65))
    B = int(rng.choice([1, 2, 3]))
    F = int(rng.choice([1, 2, 3]))
    w = int(rng.integers(5, 26)) * 8 + int(rng.integers(0, 8))
    h = int(rng.integers(4, 21)) * 8 + int(rng.integers(0, 8))
    close = float(rng.choice([0.0, 1.0]))
    route = str(rng.choice(["plain", "fused", "fused_up"]))
    extra = int(rng.choice([0, N.SPSG_FLAG_GLOBAL_MAPS, N.SPSG_FLAG_SMEM_MAPS, ALL]))
    det = bool(rng.random() < 0.5)
    return dict(C=C, B=B, F=F, w=w, h=h, close=close, route=route, extra=extra, det=det, seed=int(rng.integers(1 << 20)))


def run_case(dev, c):
    """Deterministic mode: bit-exact gradient checks on any cameras.  Default mode: the table keeps whichever 64 pixels of
    a row arrive first, so with a table the cameras are the far ones (no row over 64 pixels) and both sides of a
    comparison average the same pixels."""
    flags = (DET if c["det"] else 0) | c["extra"]
    close = c["close"] if c["det"] or c["extra"] & ALL else 0.0
    check_render(dev, c["C"], c["B"], c["F"], c["w"], c["h"], c["seed"], flags, close)
    if c["route"] == "plain":
        check_plain_grads(dev, c["C"], c["B"], c["F"], c["w"], c["h"], c["seed"], flags, close)
    else:
        check_losses(dev, c["C"], c["B"], c["F"], c["w"], c["h"], c["seed"], True, 0.2, (1.0, 1.0, 1.0),
                     flags=flags, upstream=c["route"] == "fused_up", close=close)


def check_prebuilt(dev, C):
    """sparsify_predictions(..., raycaster=m) with a C-channel semantic head: the next forward takes
    SPSG_FLAG_INDEX_PREBUILT and renders and differentiates exactly like the forward that builds its own index."""
    from spsg_b200 import sparsify
    B, F, w, h = 2, 2, 160, 128
    _, _, _, view, intr = setup(dev, B, F, w, h, 4)
    g = torch.Generator(device="cpu").manual_seed(4)
    sdf = torch.stack([torch.from_numpy(S.sdf_volume(s)[0]) for s in range(4, 4 + B)])[:, None].contiguous().to(dev)
    col = torch.rand((B, 3) + tuple(S.DIMS_ZYX), generator=g).to(dev)
    sem = torch.randn((B, C) + tuple(S.DIMS_ZYX), generator=g).to(dev)
    n = int((sdf.abs() < S.TRUNCATION).sum())
    res = []
    for prebuilt in (True, False):
        m = module(dev, B, F, w, h, n, C, DET)
        locs, v_sdf, v_col, v_sem = sparsify.sparsify_predictions(sdf, S.TRUNCATION, None, col, sem,
                                                                   raycaster=m if prebuilt else None)
        assert v_sem.shape == (n, C)
        assert torch.equal(v_sem, sem[locs[:, 3], :, locs[:, 0], locs[:, 1], locs[:, 2]])
        nrm = torch.from_numpy(D.O.voxel_normals(n)).to(dev)
        seen = []
        real = N.lib.spsg_raycast_forward_indexed

        def spy(p, *args):
            seen.append(p._obj.flags)
            return real(p, *args)
        N.lib.spsg_raycast_forward_indexed = spy
        try:
            leaves = [x.clone().requires_grad_(True) for x in (v_sdf, v_col, nrm, v_sem)]
            outs = m(locs, *leaves, view, intr)
        finally:
            N.lib.spsg_raycast_forward_indexed = real
        assert bool(seen[0] & N.SPSG_FLAG_INDEX_PREBUILT) == prebuilt
        gimg = upstream_images(m, 9)
        grads = torch.autograd.grad(outs, leaves, gimg)
        res.append([o.detach().clone() for o in outs] + [x.clone() for x in grads])
    hit = res[0][1] != NINF
    vox = (res[0][2][..., 0] - 1).long()
    assert torch.equal(bits(res[0][3][hit]), bits(res[1][3][hit])) and torch.equal(res[0][3][hit], v_sem[vox[hit]])
    for a, b in zip(*res):
        assert torch.equal(bits(a), bits(b))


# ---- the training step with C classes (ViewGuidedTrainStep(..., num_classes=C))

TRAIN_DIMS, TRAIN_W, TRAIN_H = (32, 32, 32), 80, 64


class GenC(torch.nn.Module):
    """Seeded stand-in generator (tests/test_gpu_head_formats._Generator) with a C-channel semantic head."""

    def __init__(self, C):
        super().__init__()
        self.C = C
        self.body = torch.nn.Conv3d(4, 8, 3, padding=1)
        self.bn = torch.nn.BatchNorm3d(8)
        self.head = torch.nn.Conv3d(8, 5 + C, 1)

    def forward(self, inputs, mask, pred_sdf=(True, True), pred_color=True, pred_semantic=True):
        x = torch.relu(self.bn(self.body(inputs)))
        out = self.head(x)
        sdf = inputs[:, :1].to(out.dtype) + 0.3 * torch.tanh(out[:, 1:2])
        return out[:, :1] + 3.0, sdf, torch.tanh(out[:, 2:5]), out[:, 5:5 + self.C]


def train_sample(dev, C):
    """The synthetic batch of tests/test_gpu_head_formats with its labels 0..14 re-read as C classes: 14 (unlabeled) -> C."""
    from tests.test_gpu_head_formats import _sample
    s = _sample(dev)
    s["semantics"] = torch.where(s["semantics"] >= 14, torch.full_like(s["semantics"], C), s["semantics"])
    return s


def class_weights(dev, C):
    return torch.linspace(0.5, 2.0, C, device=dev)


def train_step(dev, model, C, flags=DET):
    from spsg_b200.train_step import ViewGuidedTrainStep
    from tests.test_gpu_head_formats import _loss_util
    step = ViewGuidedTrainStep(model, _loss_util(), 2, TRAIN_DIMS, TRAIN_W, TRAIN_H, class_weights(dev, C),
                               max_num_locs_per_sample=int(np.prod(TRAIN_DIMS)), device=dev, num_classes=C)
    step.raycaster.flags |= flags
    return step


def literal_step(dev, model, C, sample, step, flags=DET):
    """The same step from the plain raycast (RaycastRGBD, autograd) and the literal PyTorch losses: one-hot to C + 1 bins,
    labels argmax(cat(render, ones)), depth / colour L1 and the C-class cross-entropy.  Returns the loss (backward done)."""
    from spsg_b200 import normals, sparsify
    lu, T = step.loss_util, step.truncation
    inputs, mask, known = sample["input"], sample["mask"], sample.get("known")
    target_sdf, target_colors = lu.compute_targets(sample["sdf"], T, True, known, sample["colors"])
    occ, out_sdf, out_col, out_sem = model(inputs, mask, pred_sdf=[True, True], pred_color=True, pred_semantic=True)
    input_occ = torch.abs(inputs[:, :1]) < (T - 0.01)
    weight = lu.compute_dense_geo_weights(target_sdf, input_occ, T, step.weight_surf_geo, step.weight_missing_geo)
    empty = torch.sigmoid(occ.detach()) < 0.5
    weight[empty] = 0
    loss = step.w["occ"] * lu.compute_geo_occ_loss(target_sdf, occ, known, weight, T) + \
        step.w["sdf"] * lu.compute_geo_loss(target_sdf, None, out_sdf, known, weight, step.logweight_sdf)
    view, intr = sample["view_matrix"], sample["images_intrinsic"]
    transform = torch.inverse(view)
    m = RaycastRGBD(2, TRAIN_DIMS, TRAIN_W, TRAIN_H, step.raycaster.depth_min, step.raycaster.depth_max,
                    step.raycaster.thresh_sample_dist, step.raycaster.ray_increment,
                    max_num_locs_per_sample=int(np.prod(TRAIN_DIMS)), device=dev, num_classes=C)
    m.flags |= flags
    with torch.no_grad():
        locs, vals = sparsify.sparsify_predictions(target_sdf, T)
        colors = target_colors[locs[:, 3], locs[:, 0], locs[:, 1], locs[:, 2], :].float() / 255.0
        tn = normals.compute_normals_sparse(locs, vals, TRAIN_DIMS, transform=transform)
        sem = sparsify.gather_dense(locs, sample["semantics"].float())
        onehot = Fn.one_hot(sem[:, 0].long(), C + 1)[..., :-1].float().contiguous()
        rs = m(locs, vals, colors.contiguous(), tn, onehot, view, intr)[3].clone()
        lab = torch.max(torch.cat((rs, torch.ones(rs.shape[:-1] + (1,), device=dev)), -1), -1)[1].to(torch.uint8)
    locs, sdf_vals, color_vals, sem_vals = sparsify.sparsify_predictions(out_sdf, T, empty, out_col, out_sem)
    nrm = normals.compute_normals_sparse(locs, sdf_vals, TRAIN_DIMS, transform=transform)
    col, dep, _, sem_img = m(locs, sdf_vals, (color_vals + 1) * 0.5, nrm, sem_vals, view, intr)
    total2d, _ = literal_losses(col, dep, sem_img, sample["images_depth"], sample["images_color"].permute(0, 2, 3, 1),
                                lab, class_weights(dev, C), step.voxelsize,
                                (step.w["depth"], step.w["color"], step.w["semantic"]))
    loss = loss + total2d
    loss.backward()
    return loss.detach()


def check_train_step(dev, C):
    """ViewGuidedTrainStep(num_classes=C) against literal_step: loss within 1e-5, generator gradients within 2e-3 of
    their norm."""
    from tests.test_gpu_head_formats import _GradOnly
    torch.manual_seed(1234)
    base = GenC(C).to(dev)
    sample = train_sample(dev, C)
    grads, lossv = [], []
    for literal in (False, True):
        model = GenC(C).to(dev)
        model.load_state_dict(base.state_dict())
        step = train_step(dev, model, C)
        if literal:
            model.zero_grad(set_to_none=True)
            loss = literal_step(dev, model, C, {k: (v.clone() if v is not None else None) for k, v in sample.items()}, step)
        else:
            loss = step({k: (v.clone() if v is not None else None) for k, v in sample.items()}, optimizer=_GradOnly(model))
            assert step.last["num_locs"] > 0
        torch.cuda.synchronize()
        lossv.append(float(loss))
        grads.append(torch.cat([p.grad.reshape(-1) for p in model.parameters()]))
    assert abs(lossv[0] - lossv[1]) <= 1e-5 * abs(lossv[1]), lossv
    _close(grads[0], grads[1], 2e-3, "C=%d generator gradient" % C)
    return lossv


def sweep(dev, cases, seed):
    rng = np.random.default_rng(seed)
    failures = []
    for _ in range(cases):
        c = case(rng)
        try:
            run_case(dev, c)
        except AssertionError as e:
            failures.append((c, str(e)[:200]))
    return failures


if __name__ == "__main__":
    cases = int(sys.argv[1]) if len(sys.argv) > 1 else 200
    seed = int(sys.argv[2]) if len(sys.argv) > 2 else 0
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    fails = sweep(dev, cases, seed)
    print("semantic-classes sweep: %d cases, %d mismatches" % (cases, len(fails)))
    for f in fails:
        print(f)
    sys.exit(1 if fails else 0)
