"""Voxel gradients of the raycast backward, every entry against the float64 gather oracle (tests/gather_oracle.py) --
at the shapes, table sizes and flags where the gather, its row clearing and the fused loss gradients can go wrong --, and
the lifetime of the gradients the autograd Functions hand out."""
import numpy as np
import pytest
import torch

from spsg_b200 import _native as N
from tests import fuzz_gather as FZ
from tests import gather_oracle as O

pytestmark = pytest.mark.gpu

NINF = -float("inf")


def _soup_case(dev, F, det, dims=(40, 24, 36), specs=((1, "noise"), (2, "blocky")), w=64, h=48, max_pix=64, focal=1.0,
               cam_seed=17, logit_scale=1.0):
    from tests.test_gpu_adversarial import _cameras
    t, n = FZ.scene(dev, dims, list(specs))
    if logit_scale != 1.0:
        t["semantic"] = t["semantic"] * logit_scale
    B = len(specs)
    view = _cameras(dims, B * F, cam_seed, dev)
    intr = FZ.intrinsics(dev, B * F, w, h, focal)
    m = FZ.raycaster(dev, B, F, dims, w, h, n, max_pix=max_pix, deterministic=det)
    return m, t, n, view, intr


@pytest.mark.parametrize("det", [False, True])
@pytest.mark.parametrize("F", [1, 2, 3, 4])
def test_plain_backward_every_entry(cuda_device, F, det):
    """Upstream images log-uniform over 1e-6 .. 1e3 with mixed signs; rows nothing hit must be exactly 0 (the oracle's
    bound there is 0).  F > 1 deterministic: bit for bit against the fp32 emulation."""
    m, t, n, view, intr = _soup_case(cuda_device, F, det)
    tab, ties = FZ.check_plain(m, t, n, F, view, intr, seed=F)
    assert (tab.cnt == 1).any(), "no voxel hit by exactly one pixel"
    assert (tab.cnt == 0).reshape(F, n).all(0).any(), "every voxel was hit: the zero rows are not tested"
    assert ties <= n * 21 // 1000


@pytest.mark.parametrize("n", [1, 31, 33, 257])
@pytest.mark.parametrize("F,det,self_clear", [(1, False, False), (1, False, True), (2, False, True), (2, True, True)])
def test_voxel_count_edges(cuda_device, n, F, det, self_clear):
    """N around the 32-voxel warps of zero_rows (partial tail warp, ballot of hit rows), with the forward's clearing and
    with the backward clearing its own rows."""
    t, n = FZ.slab(cuda_device, n)
    view = FZ.slab_cameras(cuda_device, F)
    intr = FZ.intrinsics(cuda_device, F, 40, 36, 0.8)
    m = FZ.raycaster(cuda_device, 1, F, (16, 16, 16), 40, 36, n, deterministic=det)
    if self_clear:
        FZ.check_self_clearing(m, t, n, F, view, intr, seed=n)
    else:
        tab, _ = FZ.check_plain(m, t, n, F, view, intr, seed=n)
        assert n == 1 or (tab.cnt > 0).any()


@pytest.mark.parametrize("max_pix", [1, 5, 16, 17, 32, 33, 64])
@pytest.mark.parametrize("F,det", [(1, False), (2, False), (2, True)])
def test_max_pixels_with_overflow(cuda_device, max_pix, F, det):
    """Voxels with more pixels than their table (the gather averages the registered subset) next to voxels with a few;
    table sizes at the 16-lane group boundaries of the gather."""
    t, n = FZ.slab(cuda_device, 200)
    view = FZ.slab_cameras(cuda_device, F, seed=3)
    intr = FZ.intrinsics(cuda_device, F, 96, 80, 1.2)
    m = FZ.raycaster(cuda_device, 1, F, (16, 16, 16), 96, 80, n, max_pix=max_pix, deterministic=det)
    tab, _ = FZ.check_plain(m, t, n, F, view, intr, seed=max_pix)
    assert tab.overflow.size > 0, "no voxel overflowed its table"
    FZ.check_self_clearing(m, t, n, F, view, intr, seed=max_pix + 1)


@pytest.mark.parametrize("w,h", [(37, 29), (1, 1), (3, 70), (90, 7)])
def test_widths_not_multiples_of_the_vector_width(cuda_device, w, h):
    m, t, n, view, intr = _soup_case(cuda_device, 2, False, w=w, h=h)
    FZ.check_plain(m, t, n, 2, view, intr, seed=w)


def test_empty_chunk_and_view_that_misses(cuda_device):
    """Chunk 1 has no voxels; image 1 (chunk 0, view 1) looks away from the grid."""
    from spsg_b200 import synthetic as S
    m, t, n, view, intr = _soup_case(cuda_device, 2, False, specs=((1, "noise"), None, (2, "blocky")))
    view[1] = torch.from_numpy(S.look_at((20.0, 12.0, -30.0), (20.0, 12.0, -60.0)).astype(np.float32)).to(cuda_device)
    ls = FZ.leaves(t)
    tab, _ = FZ.check_plain(m, t, n, 2, view, intr, seed=5)
    with torch.no_grad():
        out = m(t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, intr)
    assert bool((out[1][1] == NINF).all()) and bool((out[1][2:4] == NINF).all()) and bool((out[1][0] != NINF).any())
    del ls


def test_large_launch_28_warps(cuda_device):
    """2 chunks x 2 views of 384 x 352: 16 896 tiles, the forward's 28-warp instantiation on 148 SMs."""
    m, t, n, view, intr = _soup_case(cuda_device, 2, False, dims=(48, 40, 44), w=384, h=352)
    tab, _ = FZ.check_plain(m, t, n, 2, view, intr, seed=9)
    m.flags |= N.SPSG_FLAG_DETERMINISTIC_GRADS
    FZ.check_plain(m, t, n, 2, view, intr, seed=10)


def test_large_voxel_count(cuda_device):
    m, t, n, view, intr = _soup_case(cuda_device, 1, False, dims=(64, 64, 64),
                                     specs=((3, "noise"), (4, "noise"), (5, "blocky")), w=160, h=128)
    assert n > 400000
    FZ.check_plain(m, t, n, 1, view, intr, seed=11)
    FZ.check_self_clearing(m, t, n, 1, view, intr, seed=12)


def test_grid_too_large_for_shared_memory_maps(cuda_device):
    m, t, n, view, intr = _soup_case(cuda_device, 2, False, dims=(200, 120, 96), specs=((6, "blocky"),), w=120, h=90)
    FZ.check_forward_flags(m, t, view, intr, "large grid")
    FZ.check_plain(m, t, n, 2, view, intr, seed=13)


def test_axis_longer_than_fast_path(cuda_device):
    """8200 x 4 x 4 (x longest): the march maps are off, every sample takes the exact sampler."""
    from spsg_b200 import synthetic as S
    dims = (4, 4, 8200)
    t, n = FZ.scene(cuda_device, dims, [(7, "blocky")])
    mats = [S.look_at((4100.0 + 3 * k, 2.0, -8.0), (4100.0, 2.0, 2.0), up=(0.0, 1.0, 0.0)) for k in range(2)]
    view = torch.from_numpy(np.stack(mats).astype(np.float32)).to(cuda_device)
    intr = FZ.intrinsics(cuda_device, 2, 48, 40, 0.8)
    m = FZ.raycaster(cuda_device, 1, 2, dims, 48, 40, n)
    tab, _ = FZ.check_plain(m, t, n, 2, view, intr, seed=14)
    assert (tab.cnt > 0).any()


# ---------------------------------------------------------------------------------------------------------------------
# fused 2D losses
# ---------------------------------------------------------------------------------------------------------------------

TERMS = [(d, c, s) for d in (False, True) for c in (False, True) for s in (False, True)]


@pytest.mark.parametrize("terms", TERMS)
def test_fused_term_switches(cuda_device, terms):
    """Every on/off combination of the three terms; without any term, an upstream image alone feeds the objective."""
    m, t, n, view, intr = _soup_case(cuda_device, 1, False, logit_scale=50.0)
    planes = (0, 3) if not any(terms) else ()
    FZ.check_fused(m, t, n, 1, view, intr, seed=21, terms=terms, planes=planes, grad_scale=0.37)


@pytest.mark.parametrize("det", [False, True])
@pytest.mark.parametrize("F", [1, 2, 3])
@pytest.mark.parametrize("planes", [(), (0, 2), (1,), (0, 1, 2, 3)])
def test_fused_views_and_upstream_planes(cuda_device, F, det, planes):
    """Targets equal to the rendering at some pixels (zero signs), colour weights and class weights with zeros, label 14,
    logits spread to about +-100, grad_scale != 1, subsets of upstream planes."""
    m, t, n, view, intr = _soup_case(cuda_device, F, det, logit_scale=50.0)
    FZ.check_fused(m, t, n, F, view, intr, seed=30 + F, planes=planes, grad_scale=3.0)


@pytest.mark.parametrize("F,det", [(1, False), (2, False), (2, True)])
def test_fused_direct_route(cuda_device, F, det):
    """render_loss_and_voxel_grads: the same gather without autograd."""
    m, t, n, view, intr = _soup_case(cuda_device, F, det, logit_scale=50.0)
    FZ.check_fused(m, t, n, F, view, intr, seed=40 + F, grad_scale=0.37, route_="direct")


def test_fuzz_slice(cuda_device):
    assert FZ.run(cases=16, seed0=7, dev=cuda_device) == 0


# ---------------------------------------------------------------------------------------------------------------------
# gradient lifetime
# ---------------------------------------------------------------------------------------------------------------------

def _lifetime_setup(dev, F, det):
    m, t, n, view, intr = _soup_case(dev, F, det)
    g1 = FZ.upstream_grads([(2 * F, 48, 64, 3), (2 * F, 48, 64), (2 * F, 48, 64, 3), (2 * F, 48, 64, 14)], dev, 1)
    g2 = [2.0 * x for x in g1]
    return m, t, n, view, intr, g1, g2


def _plain_pass(m, t, view, intr, xs, grads, retain=False, times=1):
    out = m(t["locs"], *xs, view, intr)
    for _ in range(times):
        torch.autograd.backward(out, grads, retain_graph=retain)


def _fused_pass(m, t, view, intr, xs, grads, retain=False, times=1):
    from spsg_b200.losses import render_with_2d_losses
    total, _, imgs = render_with_2d_losses(m, t["locs"], *xs, view, intr, differentiable_images=True)
    obj = sum((i.masked_fill(i == NINF, 0.0) * g).sum() for i, g in zip(imgs, grads))
    for _ in range(times):
        obj.backward(retain_graph=retain)


PASSES = {"plain": _plain_pass, "fused": _fused_pass}
LIFETIME = [("plain", 1, False), ("plain", 2, False), ("plain", 2, True), ("fused", 1, False), ("fused", 2, False),
            ("fused", 2, True)]


def _reference(m, t, view, intr, run, grads):
    ls = FZ.leaves(t)
    run(m, t, view, intr, ls, grads)
    return [x.grad.clone() for x in ls]


def _close(got, want):
    for a, b in zip(got, want):
        torch.testing.assert_close(a, b, rtol=1e-5, atol=1e-30)


@pytest.mark.parametrize("path,F,det", LIFETIME)
def test_two_passes_accumulate(cuda_device, path, F, det):
    """Two forward / backward pairs on one module into the same leaves: g1 + g2, not 2 g2."""
    m, t, n, view, intr, g1, g2 = _lifetime_setup(cuda_device, F, det)
    run = PASSES[path]
    r1, r2 = _reference(m, t, view, intr, run, g1), _reference(m, t, view, intr, run, g2)
    ls = FZ.leaves(t)
    run(m, t, view, intr, ls, g1)
    run(m, t, view, intr, ls, g2)
    _close([x.grad for x in ls], [a + b for a, b in zip(r1, r2)])


@pytest.mark.parametrize("leaf", [True, False])
@pytest.mark.parametrize("path,F,det", LIFETIME)
def test_retained_graph_second_backward(cuda_device, path, F, det, leaf):
    """backward(retain_graph=True) twice: 2 g, with the voxel tensors as leaves and behind a non-leaf (leaf * 1.0)."""
    m, t, n, view, intr, g1, _ = _lifetime_setup(cuda_device, F, det)
    run = PASSES[path]
    r1 = _reference(m, t, view, intr, run, g1)
    ls = FZ.leaves(t)
    xs = ls if leaf else [x * 1.0 for x in ls]
    run(m, t, view, intr, xs, g1, retain=True, times=2)
    _close([x.grad for x in ls], [2 * a for a in r1])


@pytest.mark.parametrize("path,F,det", LIFETIME)
def test_leaf_grad_does_not_alias_module_buffers(cuda_device, path, F, det):
    m, t, n, view, intr, g1, _ = _lifetime_setup(cuda_device, F, det)
    ls = FZ.leaves(t)
    PASSES[path](m, t, view, intr, ls, g1)
    bufs = [m.d_depth, m.d_color, m.d_normal, m.d_semantic]
    for x, b in zip(ls, bufs):
        st = x.grad.untyped_storage().data_ptr()
        assert st != b.untyped_storage().data_ptr(), "leaf .grad shares storage with the module's d_* buffer"
    before = [x.grad.clone() for x in ls]
    with torch.no_grad():
        m(t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, intr)
    PASSES["plain"](m, t, view, intr, FZ.leaves(t), g1)  # another backward rewrites the rows
    for x, b in zip(ls, before):
        assert torch.equal(x.grad, b), "a leaf's .grad changed under a later forward / backward of the module"


@pytest.mark.parametrize("path,F,det", LIFETIME)
def test_backward_after_superseding_forward_raises(cuda_device, path, F, det):
    m, t, n, view, intr, g1, _ = _lifetime_setup(cuda_device, F, det)
    ls = FZ.leaves(t)
    if path == "plain":
        out = m(t["locs"], *ls, view, intr)
        m(t["locs"], *FZ.leaves(t), view, intr)
        with pytest.raises(RuntimeError, match="later forward"):
            torch.autograd.backward(out, g1)
    else:
        from spsg_b200.losses import render_with_2d_losses
        total, _, imgs = render_with_2d_losses(m, t["locs"], *ls, view, intr, differentiable_images=True)
        obj = sum((i.masked_fill(i == NINF, 0.0) * g).sum() for i, g in zip(imgs, g1))
        with torch.no_grad():
            m(t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, intr)
        with pytest.raises(RuntimeError, match="later forward"):
            obj.backward()
