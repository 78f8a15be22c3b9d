"""BASELINE configs[2] at full size -- 8 chunks x 5 views at 320x256 -- against the compiled reference extension.

This is the launch every C3 / room number of bench.py comes from: 131 072 warp tiles, i.e. the large-launch instantiation
of the forward kernel (`raycast_forward_kernel<*,*,kFwdWarpsLarge>`, selected from 148*4*28 = 16 576 tiles on), more than one
tile per warp, dynamic tile counters and -- in the ragged case -- work stealing across chunks.  The reference renders one
view per chunk and call, so it is looped over the five views (gradients accumulated, as autograd would)."""
import numpy as np
import pytest
import torch

from oracle import ref_driver as refdriver
from tests.common import count_bit_mismatch, scene_tensors, views

pytestmark = pytest.mark.gpu

B, F = 8, 5


def _modules(device, n, batch=B, frames=F):
    from spsg_b200 import synthetic as S
    from spsg_b200.raycast_rgbd import RaycastRGBD
    if not refdriver.available(pinned=True):
        pytest.skip("oracle/_ref not built (run __graft_entry__.build() where /root/reference exists)")
    n_max = n // batch + 1000
    mine = RaycastRGBD(batch, S.DIMS_ZYX, S.WIDTH, S.HEIGHT, S.DEPTH_MIN, S.DEPTH_MAX, S.THRESH_SAMPLE_DIST, S.RAY_INCREMENT,
                       max_num_frames=frames, max_num_locs_per_sample=n_max, device=device)
    ref = refdriver.RefRaycaster(batch, S.DIMS_ZYX, S.WIDTH, S.HEIGHT, S.DEPTH_MIN, S.DEPTH_MAX, S.THRESH_SAMPLE_DIST,
                                 S.RAY_INCREMENT, n_max, 64, device=device, pinned=True)
    return mine, ref


def _sel(f, device, batch=B, frames=F):
    return torch.arange(batch, device=device) * frames + f   # image of chunk b, view f


def test_c3_forward_and_gradients_match_looped_reference(cuda_device):
    from spsg_b200 import synthetic as S
    torch.manual_seed(3)
    _, t = scene_tensors(list(range(40, 40 + B)), cuda_device)
    n = t["locs"].shape[0]
    _, _, view, intr = views(B, F, cuda_device, seed=11)
    mine, ref = _modules(cuda_device, n)
    tiles = (S.WIDTH // 8) * (S.HEIGHT // 4) * B * F
    assert tiles >= 148 * 4 * 28, "this test must exercise the large-launch kernel instantiation"
    sdf = t["sdf"].clone().requires_grad_(True)
    col = t["color"].clone().requires_grad_(True)
    sem = t["semantic"].clone().requires_grad_(True)
    out_m = mine(t["locs"], sdf, col, t["normal"], sem, view, intr)
    assert out_m[1].shape[0] == B * F
    grads = [torch.randn_like(o) for o in out_m]
    torch.autograd.backward(out_m, grads)
    acc = [torch.zeros(n, c, device=cuda_device) for c in (3, 1, 3, 14)]
    overflow = 0
    for f in range(F):
        sel = _sel(f, cuda_device)
        out_r = ref.forward(t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view[sel].contiguous(),
                            intr[sel].contiguous())
        for name, a, b in zip(("color", "depth", "normal", "semantic"), out_m, out_r):
            assert count_bit_mismatch(a[sel], b) == 0, "view %d %s differs bitwise" % (f, name)
        assert torch.equal(mine.mapping3dto2d_num[f * n:(f + 1) * n], ref.mapping3dto2d_num[:n]), "view %d counters" % f
        overflow += int((ref.mapping3dto2d_num[:n] > 64).sum())
        d = ref.backward(*[g[sel].contiguous() for g in grads])
        for a, x in zip(acc, d):
            a += x
    assert overflow == 0  # deterministic regime: every voxel keeps all its pixels (SURVEY.md section 8(d))
    hit = out_m[1] != -float("inf")
    assert 0.4 < hit.float().mean().item() < 0.95
    for name, g, r in (("color", col.grad, acc[0]), ("sdf", sdf.grad, acc[1]), ("semantic", sem.grad, acc[3])):
        err = (g - r).abs()
        assert bool((err <= 1e-3 * r.abs() + 1e-5).all()), "%s gradients: max err %g" % (name, err.max().item())


def test_c3_fused_losses_match_literal_expressions(cuda_device):
    """The fused forward + backward pair at full C3 size against the reference's literal loss expressions applied, with
    autograd, to the un-fused rendering."""
    from oracle import losses_ref as R
    from spsg_b200 import synthetic as S
    from spsg_b200.losses import render_with_2d_losses
    _, t = scene_tensors(list(range(60, 60 + B)), cuda_device)
    n = t["locs"].shape[0]
    _, _, view, intr = views(B, F, cuda_device, seed=5)
    mine, _ = _modules(cuda_device, n)
    I = B * F
    gen = torch.Generator(device="cpu").manual_seed(9)
    t_depth = torch.where(torch.rand(I, S.HEIGHT, S.WIDTH, generator=gen) < 0.05, torch.zeros(()),
                          torch.rand(I, S.HEIGHT, S.WIDTH, generator=gen) * 0.8 + 0.8).to(cuda_device)
    t_color = torch.rand(I, S.HEIGHT, S.WIDTH, 3, generator=gen).to(cuda_device)
    t_label = torch.randint(0, 15, (I, S.HEIGHT, S.WIDTH), generator=gen, dtype=torch.uint8).to(cuda_device)
    cw = torch.tensor(S.CLASS_WEIGHTS, dtype=torch.float32, device=cuda_device)

    def leaves():
        return [t[k].clone().requires_grad_(True) for k in ("sdf", "color", "semantic")]

    sdf, col, sem = leaves()
    r_color, r_depth, _, r_sem = mine(t["locs"], sdf, col, t["normal"], sem, view, intr)
    l_depth = R.depth_l1_loss(r_depth, t_depth.unsqueeze(1), S.VOXELSIZE)
    l_color = R.compute_2dcolor_loss(r_color, t_color, None)
    l_sem = R.semantic_2d_ce_loss(r_sem, t_label.unsqueeze(-1), cw)
    (l_depth + l_color + 0.1 * l_sem).backward()
    want = [x.grad.clone() for x in (sdf, col, sem)]
    sdf, col, sem = leaves()
    total, terms, _ = render_with_2d_losses(mine, t["locs"], sdf, col, t["normal"], sem, view, intr, images_depth=t_depth,
                                            images_color=t_color, target2d_label=t_label, weight_semantic_class=cw,
                                            voxelsize=S.VOXELSIZE, weight_semantic_loss=0.1)
    total.backward()
    for got, ref in zip(terms.tolist(), (l_depth.item(), l_color.item(), l_sem.item())):
        assert abs(got - ref) <= 1e-5 * max(1.0, abs(ref)), (got, ref)
    for name, g, r in zip(("sdf", "color", "semantic"), (sdf.grad, col.grad, sem.grad), want):
        err = (g - r).abs()
        assert bool((err <= 1e-3 * r.abs() + 1e-7 + 1e-4 * r.abs().max()).all()), "%s: max err %g" % (name, err.max().item())


def test_c3_ragged_batch_work_stealing(cuda_device):
    """Half of the eight chunks hold no voxels: their CTAs run out of tiles at once and steal from the populated chunks."""
    from spsg_b200 import synthetic as S
    seeds = [70, 71, 72, 73]
    batch, t4 = scene_tensors(seeds, cuda_device)
    locs = t4["locs"].clone()
    locs[:, 3] = locs[:, 3] * 2 + 1          # the populated chunks are 1, 3, 5, 7
    t = dict(t4, locs=locs.contiguous())
    n = locs.shape[0]
    _, _, view, intr = views(B, F, cuda_device, seed=2)
    mine, ref = _modules(cuda_device, n)
    out_m = mine(t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, intr)
    for f in range(F):
        sel = _sel(f, cuda_device)
        out_r = ref.forward(t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view[sel].contiguous(),
                            intr[sel].contiguous())
        for name, a, b in zip(("color", "depth", "normal", "semantic"), out_m, out_r):
            assert count_bit_mismatch(a[sel], b) == 0, "view %d %s differs bitwise" % (f, name)
        assert torch.equal(mine.mapping3dto2d_num[f * n:(f + 1) * n], ref.mapping3dto2d_num[:n])
    depth = out_m[1].view(B, F, S.HEIGHT, S.WIDTH)
    assert bool((depth[0::2] == -float("inf")).all()) and bool((depth[1::2] != -float("inf")).any())
