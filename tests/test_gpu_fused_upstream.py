"""Fused raycast + 2D losses with differentiable renderings (render_with_2d_losses(differentiable_images=True), C ABI
spsg_raycast_backward_loss_upstream): image-space terms on the prediction's renderings (a stand-in patch discriminator)
against the un-fused route -- the module's rendering + the literal losses of oracle/losses_ref.py + autograd --, the
native composition identities, and the training step with an image loss.
Tolerances: loss values 1e-5 relative; voxel gradients 1e-3 relative (as tests/test_gpu_losses.py)."""
import types

import pytest
import torch
import torch.nn.functional as Fn

from tests.common import scene_tensors, views
from tests.fuzz_fused_upstream import close, composition, grads_of, run as fuzz_run, upstream_images

pytestmark = pytest.mark.gpu

MISS = -float("inf")


@pytest.fixture
def fp32_convolutions():
    """The stand-in discriminator's convolutions in plain fp32 (no TF32), so both routes see the same arithmetic."""
    saved = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved


def _setup(device, B, F, w, h, weight_color=False, deterministic=False):
    from oracle import losses_ref as R
    from spsg_b200 import _native as N
    from spsg_b200 import synthetic as S
    from spsg_b200.raycast_rgbd import RaycastRGBD
    seeds = list(range(20, 20 + B))
    _, pred = scene_tensors(seeds, device, payload="prediction")
    _, tgt = scene_tensors([s + 1000 for s in seeds], device, payload="target")
    n = max(pred["locs"].shape[0], tgt["locs"].shape[0])
    _, _, view, intr = views(B, F, device, seed=2, width=w, height=h)
    rc = RaycastRGBD(B, S.DIMS_ZYX, w, h, S.DEPTH_MIN, S.DEPTH_MAX, S.THRESH_SAMPLE_DIST, S.RAY_INCREMENT,
                     max_num_frames=F, max_num_locs_per_sample=n // B + 1000, device=device)
    if deterministic:
        rc.flags = N.SPSG_FLAG_DETERMINISTIC_GRADS
    with torch.no_grad():
        t_color, t_depth, _, t_sem = rc(tgt["locs"], tgt["sdf"], tgt["color"], tgt["normal"], tgt["semantic"], view, intr)
        label = R.labels_from_render(t_sem.clone())                      # (I,H,W,1) uint8
        images_depth = torch.where(t_depth != MISS, t_depth * S.VOXELSIZE, torch.zeros_like(t_depth))
        gen = torch.Generator(device="cpu").manual_seed(5)
        holes = (torch.rand(images_depth.shape, generator=gen) < 0.05).to(device)
        images_depth = images_depth.masked_fill(holes, 0.0).unsqueeze(1).contiguous()   # (I,1,H,W) like train.py:535
        images_color = torch.where(t_color != MISS, t_color, torch.full_like(t_color, 0.5)).contiguous()
    wc = None
    if weight_color:
        wc = torch.ones(B * F, 1, h, w, device=device)
        wc[:, :, : h // 2] = 3.0
    cw = torch.tensor(S.CLASS_WEIGHTS, dtype=torch.float32, device=device)
    return rc, pred, view, intr, images_depth, images_color, wc, label, cw


def _discriminator(device, channels=6, seed=11):
    """Seeded stand-in for a patch-GAN discriminator: a few convolutions, softplus mean of the patch logits."""
    g = torch.Generator().manual_seed(seed)
    net = torch.nn.Sequential(torch.nn.Conv2d(channels, 8, 4, 2, 1), torch.nn.LeakyReLU(0.2),
                              torch.nn.Conv2d(8, 8, 4, 2, 1), torch.nn.LeakyReLU(0.2), torch.nn.Conv2d(8, 1, 3, 1, 1))
    with torch.no_grad():
        for prm in net.parameters():
            prm.copy_(torch.randn(prm.shape, generator=g) * 0.3)
    net.to(device)

    def h(color, normal, cond=None):
        c = torch.where(color == MISS, torch.zeros_like(color), color * 2 - 1)
        nm = torch.where(normal == MISS, torch.zeros_like(normal), normal)
        x = torch.cat([c, nm], 3).permute(0, 3, 1, 2)
        if cond is not None:
            x = torch.cat([x, cond], 1)
        return Fn.softplus(net(x)).mean()
    return h


def _leafs(pred):
    return [pred[k].clone().requires_grad_(True) for k in ("sdf", "color", "normal", "semantic")]


def _assert_grads_close(got, want, names=("sdf", "color", "normal", "semantic")):
    for name, g, r in zip(names, got, want):
        err = (g - r).abs()
        scale = r.abs().max().item()
        assert scale > 0, name
        assert bool((err <= 1e-3 * r.abs() + 1e-6 * scale).all()), "%s: max err %g (scale %g)" % (name, err.max().item(), scale)


@pytest.mark.parametrize("B,F,weight_color", [(1, 1, False), (1, 1, True), (2, 2, False), (2, 2, True)])
def test_image_loss_matches_unfused_route(cuda_device, fp32_convolutions, B, F, weight_color):
    from oracle import losses_ref as R
    from spsg_b200 import synthetic as S
    from spsg_b200.losses import render_with_2d_losses
    w, h = 160, 128
    rc, pred, view, intr, images_depth, images_color, wc, label, cw = _setup(cuda_device, B, F, w, h, weight_color)
    disc = _discriminator(cuda_device)
    wd, wcl, ws, lam = 1.0, 0.7, 0.3, 0.5

    sdf, col, nrm, sem = _leafs(pred)
    r_color, r_depth, r_normal, r_sem = rc(pred["locs"], sdf, col, nrm, sem, view, intr)
    total = (wd * R.depth_l1_loss(r_depth, images_depth, S.VOXELSIZE) + wcl * R.compute_2dcolor_loss(r_color, images_color, wc)
             + ws * R.semantic_2d_ce_loss(r_sem, label, cw))
    obj = total + lam * disc(r_color, r_normal)
    obj.backward()
    want = [x.grad.clone() for x in (sdf, col, nrm, sem)]
    want_obj = obj.detach().clone()

    sdf2, col2, nrm2, sem2 = _leafs(pred)
    total2, _, imgs = render_with_2d_losses(
        rc, pred["locs"], sdf2, col2, nrm2, sem2, view, intr, images_depth=images_depth, images_color=images_color,
        weight_color=wc, target2d_label=label, weight_semantic_class=cw, voxelsize=S.VOXELSIZE,
        weight_depth_loss=wd, weight_color_loss=wcl, weight_semantic_loss=ws, differentiable_images=True)
    obj2 = total2 + lam * disc(imgs[0], imgs[2])
    obj2.backward()
    torch.testing.assert_close(obj2.detach(), want_obj, rtol=1e-5, atol=1e-7)
    assert float(nrm2.grad.abs().max()) > 0
    _assert_grads_close([sdf2.grad, col2.grad, nrm2.grad, sem2.grad], want)


def _forward(rc, pred, view, intr, images_depth, images_color, wc, label, cw):
    from spsg_b200 import losses as L
    from spsg_b200 import synthetic as S
    targets = (images_depth.contiguous(), images_color.contiguous(), None if wc is None else wc.contiguous(),
               label.contiguous(), cw, S.VOXELSIZE, (1.0, 0.7, 0.3))
    return L.fused_forward(rc, pred["locs"], pred["sdf"], pred["color"], pred["normal"], pred["semantic"], view, intr,
                           targets, False)


@pytest.mark.parametrize("F,deterministic", [(1, False), (2, True)])
def test_native_composition(cuda_device, F, deterministic):
    """The upstream entry point = spsg_raycast_backward_loss + spsg_raycast_backward of the same images, for all four
    planes, each plane alone and no plane at all."""
    from spsg_b200 import losses as L
    from spsg_b200 import synthetic as S
    w, h = 160, 128
    setup = _setup(cuda_device, 2, F, w, h, weight_color=True, deterministic=deterministic)
    rc, pred = setup[0], setup[1]
    n = pred["locs"].shape[0]
    p, tg, loss_out = _forward(*setup)
    scale = torch.tensor(1.7, device=cuda_device)
    gen = torch.Generator().manual_seed(3)
    for planes in ([0, 1, 2, 3], [0], [1], [2], [3], [0, 2]):
        up = upstream_images(2 * F, h, w, planes, gen, cuda_device)
        got, want = composition(rc, p, tg, loss_out, scale, up, n, S.DIMS_ZYX)
        assert close(got, want), planes
        assert float(got[2].abs().max()) > 0 or 2 not in planes
    # no plane: exactly the fused backward without upstream
    L.fused_backward(rc, p, tg, loss_out, scale, False, upstream=(None,) * 4)
    none = grads_of(rc, n)
    L.fused_backward(rc, p, tg, loss_out, scale, False)
    for a, b in zip(none, grads_of(rc, n)):
        assert torch.equal(a, b)


@pytest.mark.parametrize("F,deterministic", [(1, False), (2, True)])
def test_native_identities(cuda_device, F, deterministic):
    from spsg_b200 import losses as L
    from spsg_b200 import raycast_rgbd_cuda as rcc
    from spsg_b200 import synthetic as S
    w, h = 96, 80
    setup = _setup(cuda_device, 2, F, w, h, deterministic=deterministic)
    rc, pred = setup[0], setup[1]
    n = pred["locs"].shape[0]
    p, tg, loss_out = _forward(*setup)
    scale = torch.tensor(0.8, device=cuda_device)
    I = 2 * F
    # all-zero upstream images: bit-identical to the fused backward
    zero = upstream_images(I, h, w, [0, 1, 2, 3], torch.Generator().manual_seed(0), cuda_device)
    zero = tuple(torch.zeros_like(z) for z in zero)
    L.fused_backward(rc, p, tg, loss_out, scale, False, upstream=zero)
    a = grads_of(rc, n)
    L.fused_backward(rc, p, tg, loss_out, scale, False)
    for x, y in zip(a, grads_of(rc, n)):
        assert torch.equal(x, y)
    # loss targets off: bit-identical to the plain backward of the same images
    up = upstream_images(I, h, w, [0, 1, 2, 3], torch.Generator().manual_seed(1), cuda_device)
    L.fused_backward(rc, p, L._targets_off(tg), loss_out, None, False, upstream=up)
    a = grads_of(rc, n)
    rcc.backward(up[0], up[1], up[2], up[3], rc.sparse_mapping, rc.mapping3dto2d, rc.mapping3dto2d_num,
                 [2, S.DIMS_ZYX[2], S.DIMS_ZYX[1], S.DIMS_ZYX[0], n], rc.d_color, rc.d_depth, rc.d_normal,
                 rc.d_semantic, views_per_chunk=F, workspace_owner=rc.workspace, flags=rc.flags)
    for x, y in zip(a, grads_of(rc, n)):
        assert torch.equal(x, y)


def test_images_only_objective_with_empty_loss_sets_has_no_nan(cuda_device, fp32_convolutions):
    """Only the renderings feed the objective and the depth target is all holes (its term is NaN, like torch's mean over
    an empty set): the voxel gradients are those of the image term alone, finite."""
    from spsg_b200 import synthetic as S
    from spsg_b200.losses import render_with_2d_losses
    w, h = 96, 80
    rc, pred, view, intr, images_depth, _, _, _, _ = _setup(cuda_device, 1, 1, w, h)
    disc = _discriminator(cuda_device)
    sdf, col, nrm, sem = _leafs(pred)
    total, _, imgs = render_with_2d_losses(rc, pred["locs"], sdf, col, nrm, sem, view, intr,
                                           images_depth=torch.zeros_like(images_depth), voxelsize=S.VOXELSIZE,
                                           differentiable_images=True)
    assert torch.isnan(total)
    disc(imgs[0], imgs[2]).backward()
    got = [sdf.grad.clone(), col.grad.clone(), nrm.grad.clone()]
    for g in got:
        assert bool(torch.isfinite(g).all())
    assert float(nrm.grad.abs().max()) > 0 and float(col.grad.abs().max()) > 0
    # the same gradients through the un-fused module
    sdf2, col2, nrm2, sem2 = _leafs(pred)
    r_color, _, r_normal, _ = rc(pred["locs"], sdf2, col2, nrm2, sem2, view, intr)
    disc(r_color, r_normal).backward()
    _assert_grads_close(got[1:], [col2.grad, nrm2.grad], names=("color", "normal"))


def test_unused_differentiable_images_change_nothing(cuda_device):
    from spsg_b200 import synthetic as S
    from spsg_b200.losses import render_with_2d_losses
    w, h = 96, 80
    rc, pred, view, intr, images_depth, images_color, wc, label, cw = _setup(cuda_device, 2, 2, w, h, deterministic=True)
    out = []
    for diff in (False, True):
        leafs = _leafs(pred)
        total, _, _ = render_with_2d_losses(rc, pred["locs"], *leafs, view, intr, images_depth=images_depth,
                                            images_color=images_color, target2d_label=label, weight_semantic_class=cw,
                                            voxelsize=S.VOXELSIZE, differentiable_images=diff)
        (total * 1.3).backward()
        out.append([x.grad.clone() for x in leafs])
    for a, b in zip(*out):
        assert torch.equal(a, b)


def test_inplace_change_of_a_rendering_before_backward_raises(cuda_device):
    from spsg_b200 import synthetic as S
    from spsg_b200.losses import render_with_2d_losses
    w, h = 96, 80
    rc, pred, view, intr, images_depth, images_color, wc, label, cw = _setup(cuda_device, 1, 1, w, h)
    sdf, col, nrm, sem = _leafs(pred)
    total, _, imgs = render_with_2d_losses(rc, pred["locs"], sdf, col, nrm, sem, view, intr, images_depth=images_depth,
                                           voxelsize=S.VOXELSIZE, differentiable_images=True)
    obj = total + imgs[0].clamp(min=0).mean()
    with pytest.raises(RuntimeError):  # raised by the in-place op itself or, at the latest, by backward()
        imgs[1].mul_(2.0)
        obj.backward()
    # the module's own buffer changed in place: backward() refuses too
    sdf, col, nrm, sem = _leafs(pred)
    total, _, imgs = render_with_2d_losses(rc, pred["locs"], sdf, col, nrm, sem, view, intr, images_depth=images_depth,
                                           voxelsize=S.VOXELSIZE, differentiable_images=True)
    rc.image_depth.mul_(2.0)
    with pytest.raises(RuntimeError):
        total.backward()


def test_module_buffers_do_not_chain_graphs(cuda_device, fp32_convolutions):
    """Two steps on one module, each with its own backward: the second render does not reach into the first graph."""
    from spsg_b200 import synthetic as S
    from spsg_b200.losses import render_with_2d_losses
    w, h = 96, 80
    rc, pred, view, intr, images_depth, _, _, _, _ = _setup(cuda_device, 1, 1, w, h)
    disc = _discriminator(cuda_device)
    for _ in range(2):
        with torch.no_grad():
            rc(pred["locs"], pred["sdf"], pred["color"], pred["normal"], pred["semantic"], view, intr)
        sdf, col, nrm, sem = _leafs(pred)
        r_color, _, r_normal, _ = rc(pred["locs"], sdf, col, nrm, sem, view, intr)
        disc(r_color, r_normal).backward()
        total, _, imgs = render_with_2d_losses(rc, pred["locs"], sdf, col, nrm, sem, view, intr,
                                               images_depth=images_depth, voxelsize=S.VOXELSIZE,
                                               differentiable_images=True)
        (total + disc(imgs[0], imgs[2])).backward()
        assert not rc.image_color.requires_grad and bool(torch.isfinite(nrm.grad).all())


def test_fuzz_slice(cuda_device):
    assert fuzz_run(cases=24, seed0=5, dev=cuda_device) == 0


# ---- the training step with an image loss ------------------------------------------------------------------------

DIMS = (32, 32, 32)
W, H = 80, 64


class _Generator(torch.nn.Module):
    """Small seeded stand-in with the reference generator's call signature and dense heads."""

    def __init__(self):
        super().__init__()
        self.body = torch.nn.Conv3d(4, 8, 3, padding=1)
        self.occ, self.sdf = torch.nn.Conv3d(8, 1, 1), torch.nn.Conv3d(8, 1, 1)
        self.color, self.semantic = torch.nn.Conv3d(8, 3, 1), torch.nn.Conv3d(8, 14, 1)

    def forward(self, inputs, mask, pred_sdf=(True, True), pred_color=True, pred_semantic=True):
        x = torch.relu(self.body(inputs))
        sdf = inputs[:, :1] + 0.3 * torch.tanh(self.sdf(x))
        return self.occ(x) + 3.0, sdf, torch.tanh(self.color(x)), self.semantic(x)


def _loss_util():
    """Stand-in dense 3D losses with the reference loss module's names and signatures."""
    return types.SimpleNamespace(
        compute_targets=lambda sdf, truncation, flag, known, colors: (sdf.clone(), colors),
        compute_dense_geo_weights=lambda target, input_occ, truncation, w_surf, w_missing: torch.ones_like(target),
        compute_geo_occ_loss=lambda target, occ, known, weight, truncation: Fn.binary_cross_entropy_with_logits(
            occ, (target.abs() < truncation).float(), weight=weight),
        compute_geo_loss=lambda target, unused, sdf, known, weight, logweight: (weight * (sdf - target).abs()).mean())


def _unfused_step(model, lu, sample, cw, h, T=3.0):
    """ViewGuidedTrainStep's data flow, written out with the un-fused ops: RaycastRGBD renders, losses_2d, the image
    loss on the prediction's renderings, autograd."""
    from spsg_b200 import normals, sparsify
    from spsg_b200.losses import labels_from_render, losses_2d
    from spsg_b200.raycast_rgbd import RaycastRGBD
    B = sample["input"].shape[0]
    rc = RaycastRGBD(B, DIMS, W, H, depth_min=0.1 / 0.02, depth_max=6.0 / 0.02, thresh_sample_dist=50.5 * 0.3 * T,
                     ray_increment=0.3 * T, max_num_locs_per_sample=int(DIMS[0] * DIMS[1] * DIMS[2]))
    inputs, mask = sample["input"], sample["mask"]
    tsdf, tcol = lu.compute_targets(sample["sdf"], T, True, None, sample["colors"])
    occ, sdf, col, sem = model(inputs, mask, pred_sdf=[True, True], pred_color=True, pred_semantic=True)
    weight = lu.compute_dense_geo_weights(tsdf, torch.abs(inputs[:, :1]) < (T - 0.01), T, 1.0, 5.0)
    empty = torch.sigmoid(occ.detach()) < 0.5
    weight[empty] = 0
    loss = 1.0 * lu.compute_geo_occ_loss(tsdf, occ, None, weight, T) + 0.1 * lu.compute_geo_loss(tsdf, None, sdf, None, weight, True)
    view, intr = sample["view_matrix"], sample["images_intrinsic"]
    transform = torch.inverse(view)
    locs, vals, cols = sparsify.sparsify_predictions(inputs[:, :1].contiguous(), T, None, inputs[:, 1:4].contiguous())
    rcol, _, rnrm, _ = rc(locs, vals, cols, normals.compute_normals_sparse(locs, vals, DIMS, transform=transform), None,
                          view, intr)
    input2d = rcol.clone() * 2 - 1
    input2d[rcol == MISS] = 0
    nrm = rnrm.clone()
    nrm[rnrm == MISS] = 0
    input2d = torch.cat([input2d, nrm], 3).permute(0, 3, 1, 2).contiguous()
    with torch.no_grad():
        tl, tv = sparsify.sparsify_predictions(tsdf, T)
        tc = tcol[tl[:, 3], tl[:, 0], tl[:, 1], tl[:, 2], :].float() / 255.0
        ts = sparsify.gather_dense(tl, sample["semantics"].float())
        onehot = Fn.one_hot(ts[:, 0].long(), 15)[..., :-1].float().contiguous()
        _, _, _, tsem = rc(tl, tv, tc.contiguous(), normals.compute_normals_sparse(tl, tv, DIMS, transform=transform),
                           onehot, view, intr)
        label = labels_from_render(tsem)
    locs, sv, cv, semv = sparsify.sparsify_predictions(sdf, T, empty, col, sem)
    onrm = normals.compute_normals_sparse(locs, sv, DIMS, transform=transform)
    r = rc(locs, sv, (cv + 1) * 0.5, onrm, semv, view, intr)
    total2d, _ = losses_2d(r[0], r[1], r[3], images_depth=sample["images_depth"],
                           images_color=sample["images_color"].permute(0, 2, 3, 1), target2d_label=label,
                           weight_semantic_class=cw, voxelsize=0.02, weight_depth_loss=1.0, weight_color_loss=1.0,
                           weight_semantic_loss=0.1)
    loss = loss + total2d + h(r, input2d)
    loss.backward()
    return float(loss.detach())


def test_train_step_with_image_loss_matches_unfused_composition(cuda_device, fp32_convolutions):
    from spsg_b200 import synthetic as S
    from spsg_b200.train_step import ViewGuidedTrainStep
    torch.manual_seed(1234)
    model = _Generator().to(cuda_device)
    sample = S.make_train_sample([0, 1], 1, dims_zyx=DIMS, width=W, height=H,
                                 view_kw=dict(center=(16.0, 16.0, 14.0), radius=38.0, height=30.0))
    sample = {k: torch.from_numpy(v).to(cuda_device) for k, v in sample.items()}
    sample["known"] = None
    cw = torch.tensor(S.CLASS_WEIGHTS, dtype=torch.float32, device=cuda_device)
    disc = _discriminator(cuda_device, channels=12)
    seen = {}

    def image_loss(pred, input2d):
        seen["input2d"] = None if input2d is None else input2d.clone()
        return 0.5 * disc(pred[0], pred[2], input2d)

    class _Opt:
        def zero_grad(self, set_to_none=True):
            model.zero_grad(set_to_none=True)

        def step(self):
            pass

    step = ViewGuidedTrainStep(model, _loss_util(), 2, DIMS, W, H, cw, max_num_locs_per_sample=int(DIMS[0] * DIMS[1] * DIMS[2]),
                               device=cuda_device, image_loss=image_loss)
    render_input = step._render_input

    def render_input_and_clone(*args):
        c, nm = render_input(*args)
        seen["input_render"] = (c.clone(), nm.clone())
        return c, nm
    step._render_input = render_input_and_clone
    loss = float(step({k: (v.clone() if v is not None else None) for k, v in sample.items()}, optimizer=_Opt()))
    torch.cuda.synchronize()
    got = torch.cat([q.grad.reshape(-1) for q in model.parameters()])
    assert step.last["num_locs"] > 1000 and torch.isfinite(step.last["image_loss"])
    c, nm = seen["input_render"]
    want2d = torch.cat([torch.where(c == MISS, torch.zeros_like(c), c * 2 - 1),
                        torch.where(nm == MISS, torch.zeros_like(nm), nm)], 3).permute(0, 3, 1, 2).contiguous()
    assert torch.equal(seen["input2d"], want2d)

    model.zero_grad(set_to_none=True)
    loss_r = _unfused_step(model, _loss_util(), sample, cw, lambda r, x: 0.5 * disc(r[0], r[2], x))
    want = torch.cat([q.grad.reshape(-1) for q in model.parameters()])
    assert abs(loss - loss_r) <= 1e-5 * max(1.0, abs(loss_r)), (loss, loss_r)
    rel = float((got - want).norm() / want.norm())
    assert rel < 2e-3, rel
