"""Per-view normals for renders with several views per chunk (SPSG_FLAG_VIEW_NORMALS): the normals op
(``compute_normals_sparse(..., views_per_chunk=F)``, ``spsg_normals_*_views``), the raycast forward and backward against
per-view single launches, autograd end to end, the training step with F = 2, validation, and a slice of
tests/fuzz_view_normals.py."""
import types

import numpy as np
import pytest
import torch
import torch.nn.functional as Fn

from spsg_b200 import _native as N
from tests import fuzz_gather as FZ
from tests import fuzz_view_normals as VN
from tests.common import scene_tensors, views

pytestmark = pytest.mark.gpu

MISS = -float("inf")


def _synthetic(dev, B, F, w=320, h=256, seed=0):
    from spsg_b200 import synthetic as S
    from spsg_b200.raycast_rgbd import RaycastRGBD
    _, t = scene_tensors(list(range(30 + seed, 30 + seed + B)), dev)
    n = t["locs"].shape[0]
    _, _, view, intr = views(B, F, dev, seed=3 + seed, width=w, height=h)

    def module(frames):
        return RaycastRGBD(B, S.DIMS_ZYX, w, h, S.DEPTH_MIN, S.DEPTH_MAX, S.THRESH_SAMPLE_DIST, S.RAY_INCREMENT,
                           max_num_frames=frames, max_num_locs_per_sample=n // B + 1000, device=dev)
    return t, n, view, intr, module


# ---- 1, 2: the normals op ------------------------------------------------------------------------------------------

@pytest.mark.parametrize("F", [1, 2, 3, 5])
def test_normals_op_forward_matches_per_view_calls(cuda_device, F):
    from spsg_b200 import synthetic as S
    from spsg_b200.normals import compute_normals_sparse
    B = 3
    _, t = scene_tensors([7, 8, 9], cuda_device)
    _, _, view, _ = views(B, F, cuda_device, seed=4)
    T = torch.inverse(view)
    out = compute_normals_sparse(t["locs"], t["sdf"], S.DIMS_ZYX, transform=T, views_per_chunk=F)
    n = t["locs"].shape[0]
    assert tuple(out.shape) == ((n, 3) if F == 1 else (n, F, 3))
    out = out.reshape(n, F, 3)
    for f in range(F):
        want = compute_normals_sparse(t["locs"], t["sdf"], S.DIMS_ZYX, transform=T[f::F].contiguous(), num_chunks=B)
        assert torch.equal(out[:, f].contiguous().view(torch.int32), want.view(torch.int32)), f
    assert bool((out.abs().sum(-1) > 0).any())


@pytest.mark.parametrize("F", [1, 2, 3, 5])
def test_normals_op_backward_matches_per_view_calls(cuda_device, F):
    """d_sdf against autograd through the F separate calls.  The per-view terms of u = dL/dg are the same fp32 values; here
    they are summed over the views first and then gathered from the six neighbours, there gathered per view and summed by
    autograd: the two differ by reassociation of at most 6 F terms, bounded here by 2^-20 * F * (|d_sdf| + max|d_sdf|)."""
    from spsg_b200 import synthetic as S
    from spsg_b200.normals import compute_normals_sparse
    B = 2
    _, t = scene_tensors([11, 12], cuda_device)
    _, _, view, _ = views(B, F, cuda_device, seed=5)
    T = torch.inverse(view)
    n = t["locs"].shape[0]
    g = torch.Generator(device="cpu").manual_seed(F)
    up = torch.randn((n, F, 3), generator=g).to(cuda_device)
    x = t["sdf"].clone().requires_grad_(True)
    out = compute_normals_sparse(t["locs"], x, S.DIMS_ZYX, transform=T, views_per_chunk=F)
    (out.reshape(n, F, 3) * up).sum().backward()
    got = x.grad.clone()
    y = t["sdf"].clone().requires_grad_(True)
    for f in range(F):
        o = compute_normals_sparse(t["locs"], y, S.DIMS_ZYX, transform=T[f::F].contiguous(), num_chunks=B)
        (o * up[:, f]).sum().backward()
    want = y.grad
    assert float(want.abs().max()) > 0
    if F == 1:
        assert torch.equal(got.view(torch.int32), want.view(torch.int32))
        return
    bound = 2.0 ** -20 * F * (want.abs() + float(want.abs().max()))
    err = (got - want).abs()
    assert bool((err <= bound).all()), float((err - bound).max())


def test_normals_op_validation(cuda_device):
    from spsg_b200 import synthetic as S
    from spsg_b200.normals import compute_normals_sparse
    _, t = scene_tensors([1], cuda_device)
    with pytest.raises(RuntimeError):
        compute_normals_sparse(t["locs"], t["sdf"], S.DIMS_ZYX, views_per_chunk=2)
    with pytest.raises(RuntimeError):
        compute_normals_sparse(t["locs"], t["sdf"], S.DIMS_ZYX, transform=torch.eye(4, device=cuda_device)[None],
                               views_per_chunk=0)
    with pytest.raises(RuntimeError):  # 3 transforms for 2 chunks x 2 views
        compute_normals_sparse(t["locs"], t["sdf"], S.DIMS_ZYX, num_chunks=2,
                               transform=torch.eye(4, device=cuda_device).repeat(3, 1, 1), views_per_chunk=2)


# ---- 3, 4: the raycaster against single-view launches --------------------------------------------------------------

@pytest.mark.parametrize("fused", [False, True])
@pytest.mark.parametrize("F", [2, 3, 5])
@pytest.mark.parametrize("B", [1, 3, 8])
def test_forward_matches_single_view_launches(cuda_device, B, F, fused):
    """B = 1: maps staged in shared memory; B > 1: global maps.  B = 1, F = 2 takes the 24-warp CTA, B = 8 the 28-warp one."""
    t, n, view, intr, module = _synthetic(cuda_device, B, F, seed=B)
    m, s = module(F), module(1)
    VN.check_case(cuda_device, t, n, B, F, view, intr, m, s, "fused" if fused else "plain", seed=B * 10 + F,
                  backward=False, what="B=%d F=%d" % (B, F))


@pytest.mark.parametrize("det", [False, True])
@pytest.mark.parametrize("variant", VN.VARIANTS)
def test_backward_matches_single_view_backwards(cuda_device, variant, det):
    from tests.test_gpu_adversarial import _cameras
    dims = (40, 24, 36)
    B, F = 3, 3
    t, n = FZ.scene(cuda_device, dims, [(1, "noise"), (2, "blocky"), (3, "special")])
    view = _cameras(dims, B * F, 17, cuda_device)
    intr = FZ.intrinsics(cuda_device, B * F, 64, 48)
    m, s = VN.raycasters(cuda_device, B, F, dims, 64, 48, n, max_pix=16, det=det)
    _, ties = VN.check_case(cuda_device, t, n, B, F, view, intr, m, s, variant, seed=3)
    assert ties <= n * F * 3 // 1000


def test_backward_synthetic_c3_shape(cuda_device):
    """8 chunks x 5 views at 320 x 256 (the 28-warp forward), deterministic fused + upstream."""
    B, F = 8, 5
    t, n, view, intr, module = _synthetic(cuda_device, B, F)
    m, s = module(F), module(1)
    m.flags = N.SPSG_FLAG_DETERMINISTIC_GRADS
    VN.check_case(cuda_device, t, n, B, F, view, intr, m, s, "fused_up", seed=9)


# ---- 5: autograd end to end ----------------------------------------------------------------------------------------

def test_autograd_end_to_end_matches_single_view_composition(cuda_device):
    """Per-view normals from the normals op, rendered by render_with_2d_losses with an image term on the normal rendering:
    d vals_sdf (through the renders' depth and the normals op) and d vals_color against F single-view renders with their
    own transforms, concatenated in image order, losses_2d and the same image term."""
    from spsg_b200 import synthetic as S
    from spsg_b200.losses import losses_2d, render_with_2d_losses
    from spsg_b200.normals import compute_normals_sparse
    from tests.test_gpu_fused_upstream import _assert_grads_close, _discriminator, _setup
    saved = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        B, F, w, h = 2, 3, 160, 128
        rc, pred, view, intr, images_depth, images_color, _, label, cw = _setup(cuda_device, B, F, w, h)
        disc = _discriminator(cuda_device)
        T = torch.inverse(view)
        kw = dict(images_depth=images_depth, images_color=images_color, target2d_label=label, weight_semantic_class=cw,
                  voxelsize=S.VOXELSIZE, weight_depth_loss=1.0, weight_color_loss=0.7, weight_semantic_loss=0.3)

        sdf = pred["sdf"].clone().requires_grad_(True)
        col = pred["color"].clone().requires_grad_(True)
        nrm = compute_normals_sparse(pred["locs"], sdf, S.DIMS_ZYX, transform=T, views_per_chunk=F)
        total, _, imgs = render_with_2d_losses(rc, pred["locs"], sdf, col, nrm, pred["semantic"], view, intr,
                                               differentiable_images=True, **kw)
        obj = total + 0.5 * disc(imgs[0], imgs[2])
        obj.backward()

        sdf2 = pred["sdf"].clone().requires_grad_(True)
        col2 = pred["color"].clone().requires_grad_(True)
        from spsg_b200.raycast_rgbd import RaycastRGBD
        renders = []
        for f in range(F):
            m = RaycastRGBD(B, S.DIMS_ZYX, w, h, S.DEPTH_MIN, S.DEPTH_MAX, S.THRESH_SAMPLE_DIST, S.RAY_INCREMENT,
                            max_num_locs_per_sample=rc.max_num_locs_per_sample, device=cuda_device)
            nf = compute_normals_sparse(pred["locs"], sdf2, S.DIMS_ZYX, transform=T[f::F].contiguous(), num_chunks=B)
            renders.append(m(pred["locs"], sdf2, col2, nf, pred["semantic"], view[f::F].contiguous(),
                             intr[f::F].contiguous()))
        cat = [torch.stack([r[k] for r in renders], 1).reshape((B * F,) + tuple(renders[0][k].shape[1:]))
               for k in range(4)]
        total2, _ = losses_2d(cat[0], cat[1], cat[3], **kw)
        obj2 = total2 + 0.5 * disc(cat[0], cat[2])
        obj2.backward()
        torch.testing.assert_close(obj.detach(), obj2.detach(), rtol=1e-5, atol=1e-7)
        _assert_grads_close([sdf.grad, col.grad], [sdf2.grad, col2.grad], names=("sdf", "color"))
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved


# ---- 6: the training step with two views per chunk -----------------------------------------------------------------

def _unfused_views_step(model, lu, sample, cw, image_loss, F, T=3.0):
    """ViewGuidedTrainStep's data flow with F views per chunk, written out with single-view renders: each view's input
    and prediction normals rotated by its own camera (train.py:542-544 per reference call), renders concatenated in image
    order, losses_2d, the image loss, autograd."""
    from spsg_b200 import normals, sparsify
    from spsg_b200.losses import labels_from_render, losses_2d
    from spsg_b200.raycast_rgbd import RaycastRGBD
    from tests.test_gpu_fused_upstream import DIMS, H, W
    B = sample["input"].shape[0]

    def module(frames):
        return RaycastRGBD(B, DIMS, W, H, depth_min=0.1 / 0.02, depth_max=6.0 / 0.02, thresh_sample_dist=50.5 * 0.3 * T,
                           ray_increment=0.3 * T, max_num_frames=frames,
                           max_num_locs_per_sample=int(DIMS[0] * DIMS[1] * DIMS[2]))

    def cat(imgs):
        return torch.stack(imgs, 1).reshape((B * F,) + tuple(imgs[0].shape[1:]))

    inputs, mask = sample["input"], sample["mask"]
    tsdf, tcol = lu.compute_targets(sample["sdf"], T, True, None, sample["colors"])
    occ, sdf, col, sem = model(inputs, mask, pred_sdf=[True, True], pred_color=True, pred_semantic=True)
    weight = lu.compute_dense_geo_weights(tsdf, torch.abs(inputs[:, :1]) < (T - 0.01), T, 1.0, 5.0)
    empty = torch.sigmoid(occ.detach()) < 0.5
    weight[empty] = 0
    loss = 1.0 * lu.compute_geo_occ_loss(tsdf, occ, None, weight, T) + 0.1 * lu.compute_geo_loss(tsdf, None, sdf, None, weight, True)
    view, intr = sample["view_matrix"], sample["images_intrinsic"]
    transform = torch.inverse(view)
    vf = [view[f::F].contiguous() for f in range(F)]
    inf = [intr[f::F].contiguous() for f in range(F)]
    tf = [transform[f::F].contiguous() for f in range(F)]
    locs, vals, cols = sparsify.sparsify_predictions(inputs[:, :1].contiguous(), T, None, inputs[:, 1:4].contiguous())
    rcol, rnrm = [], []
    for f in range(F):
        r = module(1)(locs, vals, cols, normals.compute_normals_sparse(locs, vals, DIMS, transform=tf[f]), None, vf[f],
                      inf[f])
        rcol.append(r[0].clone())
        rnrm.append(r[2].clone())
    rcol, rnrm = cat(rcol), cat(rnrm)
    input2d = torch.cat([torch.where(rcol == MISS, torch.zeros_like(rcol), rcol * 2 - 1),
                         torch.where(rnrm == MISS, torch.zeros_like(rnrm), rnrm)], 3).permute(0, 3, 1, 2).contiguous()
    with torch.no_grad():
        tl, tv = sparsify.sparsify_predictions(tsdf, T)
        tc = tcol[tl[:, 3], tl[:, 0], tl[:, 1], tl[:, 2], :].float() / 255.0
        ts = sparsify.gather_dense(tl, sample["semantics"].float())
        onehot = Fn.one_hot(ts[:, 0].long(), 15)[..., :-1].float().contiguous()
        _, _, _, tsem = module(F)(tl, tv, tc.contiguous(), normals.compute_normals_sparse(tl, tv, DIMS, num_chunks=B),
                                  onehot, view, intr)
        label = labels_from_render(tsem)
    locs, sv, cv, semv = sparsify.sparsify_predictions(sdf, T, empty, col, sem)
    rs = []
    for f in range(F):
        onrm = normals.compute_normals_sparse(locs, sv, DIMS, transform=tf[f])
        rs.append(module(1)(locs, sv, (cv + 1) * 0.5, onrm, semv, vf[f], inf[f]))
    r = [cat([x[k] for x in rs]) for k in range(4)]
    total2d, _ = losses_2d(r[0], r[1], r[3], images_depth=sample["images_depth"],
                           images_color=sample["images_color"].permute(0, 2, 3, 1), target2d_label=label,
                           weight_semantic_class=cw, voxelsize=0.02, weight_depth_loss=1.0, weight_color_loss=1.0,
                           weight_semantic_loss=0.1)
    loss = loss + total2d + image_loss(r, input2d)
    loss.backward()
    return float(loss.detach()), input2d.detach()


def test_train_step_two_views_matches_per_view_composition(cuda_device):
    """With F = 2 the step renders the input scan and the prediction with per-view normals: input2d's normal channels
    are bit-identical to per-view single renders, loss and generator gradients match the per-view un-fused route.
    (Before per-view normals, every chunk b was rotated by image b's camera -- a camera of another chunk for b >= 1.)"""
    from spsg_b200 import synthetic as S
    from spsg_b200.train_step import ViewGuidedTrainStep
    from tests.test_gpu_fused_upstream import DIMS, H, W, _Generator, _discriminator, _loss_util
    saved = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        F = 2
        torch.manual_seed(1234)
        model = _Generator().to(cuda_device)
        sample = S.make_train_sample([0, 1], F, dims_zyx=DIMS, width=W, height=H,
                                     view_kw=dict(center=(16.0, 16.0, 14.0), radius=38.0, height=30.0))
        sample = {k: torch.from_numpy(v).to(cuda_device) for k, v in sample.items()}
        sample["known"] = None
        cw = torch.tensor(S.CLASS_WEIGHTS, dtype=torch.float32, device=cuda_device)
        disc = _discriminator(cuda_device, channels=12)
        seen = {}

        def image_loss(pred, input2d):
            seen["input2d"] = input2d.clone()
            return 0.5 * disc(pred[0], pred[2], input2d)

        opt = types.SimpleNamespace(zero_grad=lambda set_to_none=True: model.zero_grad(set_to_none=True),
                                    step=lambda: None)
        step = ViewGuidedTrainStep(model, _loss_util(), 2, DIMS, W, H, cw, views_per_chunk=F,
                                   max_num_locs_per_sample=int(DIMS[0] * DIMS[1] * DIMS[2]), device=cuda_device,
                                   image_loss=image_loss)
        loss = float(step({k: (v.clone() if v is not None else None) for k, v in sample.items()}, optimizer=opt))
        torch.cuda.synchronize()
        got = torch.cat([q.grad.reshape(-1) for q in model.parameters()])
        assert step.last["num_locs"] > 1000 and torch.isfinite(step.last["image_loss"])

        model.zero_grad(set_to_none=True)
        loss_r, input2d_r = _unfused_views_step(model, _loss_util(), sample, cw,
                                                lambda r, x: 0.5 * disc(r[0], r[2], x), F)
        want = torch.cat([q.grad.reshape(-1) for q in model.parameters()])
        assert torch.equal(seen["input2d"][:, 3:].contiguous().view(torch.int32),
                           input2d_r[:, 3:].contiguous().view(torch.int32))
        assert torch.equal(seen["input2d"], input2d_r)
        assert abs(loss - loss_r) <= 1e-5 * max(1.0, abs(loss_r)), (loss, loss_r)
        rel = float((got - want).norm() / want.norm())
        assert rel < 2e-3, rel
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved


# ---- 7: validation, mode mismatch, gradient accumulation ----------------------------------------------------------

def _small(dev, F=3, det=False):
    from tests.test_gpu_adversarial import _cameras
    dims = (24, 20, 28)
    t, n = FZ.scene(dev, dims, [(1, "noise"), (2, "blocky")])
    view = _cameras(dims, 2 * F, 5, dev)
    intr = FZ.intrinsics(dev, 2 * F, 48, 40)
    m = FZ.raycaster(dev, 2, F, dims, 48, 40, n, deterministic=det)
    P = VN.view_payload(n, F, dev, np.random.default_rng(0))
    return m, t, n, view, intr, P


def _stable_rows(m, n, F):
    """(N,F) True where the (voxel, view) table did not overflow: only those means are the same from pass to pass (an
    overflowing voxel keeps whichever max_pixels_per_voxel pixels registered first)."""
    return (m.mapping3dto2d_num[:F * n].view(F, n) <= m.mapping3dto2d.shape[1]).t()


def test_wrong_view_count_raises(cuda_device):
    from spsg_b200 import synthetic as S
    from spsg_b200.losses import render_loss_and_voxel_grads, render_with_2d_losses
    m, t, n, view, intr, P = _small(cuda_device, F=3)
    for bad in (P[:, :2].contiguous(), torch.zeros(n, 4, 3, device=cuda_device), torch.zeros(n, 3, 2, device=cuda_device)):
        with pytest.raises(RuntimeError):
            m(t["locs"], t["sdf"], t["color"], bad, t["semantic"], view, intr)
        with pytest.raises(RuntimeError):
            render_with_2d_losses(m, t["locs"], t["sdf"], t["color"], bad, t["semantic"], view, intr,
                                  voxelsize=S.VOXELSIZE)
        with pytest.raises(RuntimeError):
            render_loss_and_voxel_grads(m, t["locs"], t["sdf"], t["color"], bad, t["semantic"], view, intr)


def test_backward_in_the_other_mode_raises(cuda_device):
    from spsg_b200 import raycast_rgbd_cuda as rcc
    m, t, n, view, intr, P = _small(cuda_device, F=3)
    dims = [2, m.dims3d[2], m.dims3d[1], m.dims3d[0], n]
    for per_view in (True, False):
        with torch.no_grad():
            out = m(t["locs"], t["sdf"], t["color"], P if per_view else P[:, 0].contiguous(), t["semantic"], view, intr)
        grads = [torch.ones_like(o) for o in out]
        other = 0 if per_view else N.SPSG_FLAG_VIEW_NORMALS
        with pytest.raises(RuntimeError, match="without a matching forward"):
            rcc.backward(*grads, m.sparse_mapping, m.mapping3dto2d, m.mapping3dto2d_num, dims, m.d_color, m.d_depth,
                         rcc.normal_grad_buffer(m, not per_view), m.d_semantic, views_per_chunk=3,
                         workspace_owner=m.workspace, flags=other)


@pytest.mark.parametrize("path", ["plain", "fused"])
@pytest.mark.parametrize("det", [False, True])
def test_leaf_grad_accumulates_over_two_passes(cuda_device, path, det):
    from spsg_b200 import synthetic as S
    from spsg_b200.losses import render_with_2d_losses
    m, t, n, view, intr, P = _small(cuda_device, F=3, det=det)
    gen = torch.Generator().manual_seed(2)

    def one(x, k):
        if path == "plain":
            out = m(t["locs"], t["sdf"], t["color"], x, t["semantic"], view, intr)
            g = torch.randn(out[2].shape, generator=gen).to(cuda_device)
            torch.autograd.backward(out[2], g)
        else:
            total, _, imgs = render_with_2d_losses(m, t["locs"], t["sdf"], t["color"], x, t["semantic"], view, intr,
                                                   voxelsize=S.VOXELSIZE, differentiable_images=True)
            g = torch.randn(imgs[2].shape, generator=gen).to(cuda_device)
            (imgs[2].masked_fill(imgs[2] == MISS, 0.0) * g).sum().backward()

    gen.manual_seed(2)
    singles = []
    for k in range(2):
        x = P.clone().requires_grad_(True)
        one(x, k)
        singles.append(x.grad.clone())
    gen.manual_seed(2)
    x = P.clone().requires_grad_(True)
    one(x, 0)
    one(x, 1)
    assert tuple(x.grad.shape) == (n, 3, 3)
    assert float(singles[0].abs().max()) > 0
    keep = _stable_rows(m, n, 3)
    assert bool(keep.any())
    # (rtol: each pass re-registers its pixels, so a near-tie may round the other way; aliasing would give 2 * g2)
    torch.testing.assert_close(x.grad[keep], (singles[0] + singles[1])[keep], rtol=1e-6, atol=0)


def test_shared_normals_unchanged_by_the_views_buffer(cuda_device):
    """(N,3) normals keep using d_normal: a per-view pass before does not alter a shared pass's gradients."""
    m, t, n, view, intr, P = _small(cuda_device, F=3, det=True)
    res = []
    for warm in (False, True):
        if warm:
            x = P.clone().requires_grad_(True)
            out = m(t["locs"], t["sdf"], t["color"], x, t["semantic"], view, intr)
            torch.autograd.backward(out[2], torch.ones_like(out[2]))
        y = P[:, 0].clone().requires_grad_(True)
        out = m(t["locs"], t["sdf"], t["color"], y, t["semantic"], view, intr)
        torch.autograd.backward(out[2], torch.ones_like(out[2]))
        res.append(y.grad.clone())
        assert tuple(y.grad.shape) == (n, 3)
    keep = _stable_rows(m, n, 3).all(1)
    assert bool(keep.any())
    torch.testing.assert_close(res[1][keep], res[0][keep], rtol=1e-6, atol=0)


# ---- 8: fuzz slice -------------------------------------------------------------------------------------------------

def test_fuzz_slice(cuda_device):
    assert VN.run(cases=30, seed0=3, dev=cuda_device) == 0
