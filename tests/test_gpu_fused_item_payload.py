"""The fused gather reads each (voxel, view) item's logits and colour once, from its first registered pixel, and forms the
softmax once per item.  Here it is checked bit for bit against the per-pixel route over the same renderings and tables:
the gradient images of spsg_losses2d_backward (the per-pixel loss gradients, computed with the forward's normalisers)
gathered by the plain backward.  Both sum the same fp32 terms in the same registration order, so with one view per chunk
or SPSG_FLAG_DETERMINISTIC_GRADS every voxel gradient must agree exactly.  The payload carries what a per-item read has
to treat as the per-pixel one does: NaN and +-inf logits, -inf in logit 0 (no semantic term), -inf and NaN colour
channels; the targets mix label 14 into items, give a colour weight with zeros, and, optionally, upstream images."""
import ctypes

import numpy as np
import pytest
import torch

from spsg_b200 import _native as N
from tests import fuzz_gather as FZ
from tests.test_gpu_gather_oracle import _soup_case

pytestmark = pytest.mark.gpu

NINF = -float("inf")


def _poison_payload(t, seed):
    """Voxel rows with special logits and colours, a few percent of each kind."""
    g = torch.Generator().manual_seed(seed)
    sem, col = t["semantic"].clone(), t["color"].clone()
    n = sem.shape[0]
    pick = lambda frac: torch.nonzero(torch.rand(n, generator=g) < frac)[:, 0].to(sem.device)
    chan = lambda rows, lo=0: torch.randint(lo, 14, (rows.numel(),), generator=g).to(sem.device)
    r = pick(0.03); sem[r, chan(r)] = float("nan")
    r = pick(0.03); sem[r, chan(r)] = float("inf")
    r = pick(0.03); sem[r, chan(r, 1)] = NINF
    r = pick(0.03); sem[r, 0] = NINF
    r = pick(0.01); sem[r] = float("nan")
    r = pick(0.03); col[r, torch.randint(0, 3, (r.numel(),), generator=g).to(sem.device)] = NINF
    r = pick(0.02); col[r, torch.randint(0, 3, (r.numel(),), generator=g).to(sem.device)] = float("nan")
    t = dict(t)
    t["semantic"], t["color"] = sem.contiguous(), col.contiguous()
    return t


def _same(a, b):
    """Bit for bit, NaN where the other has NaN (its payload bits aside)."""
    na, nb = torch.isnan(a), torch.isnan(b)
    if not torch.equal(na, nb):
        return False
    return torch.equal(a.masked_fill(na, 0).view(torch.int32), b.masked_fill(nb, 0).view(torch.int32))


@pytest.mark.parametrize("upstream", [False, True])
@pytest.mark.parametrize("F,det", [(1, False), (2, True), (3, True)])
def test_fused_gather_matches_per_pixel_route(cuda_device, F, det, upstream):
    from spsg_b200 import losses as L
    from spsg_b200 import raycast_rgbd_cuda as rc
    dev = cuda_device
    m, t, n, view, intr = _soup_case(dev, F, det, logit_scale=50.0)
    t = _poison_payload(t, 100 + F)
    rng = np.random.default_rng(200 + F)
    with torch.no_grad():
        pre = [o.clone() for o in m(t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, intr)]
    tg, _ = FZ.fused_targets(pre, rng, dev)
    assert tg["weight_color"] is not None and bool((tg["target2d_label"] == 14).any())
    I = view.shape[0]
    ups = None
    if upstream:
        gc, _, _, gs = FZ.upstream_grads([(I, m.height, m.width, 3), (1,), (1,), (I, m.height, m.width, 14)], dev, 300 + F)
        ups = (gc, None, None, gs)
    scale = torch.tensor(0.37, device=dev)
    targets = (tg["images_depth"], tg["images_color"], tg["weight_color"], tg["target2d_label"],
               tg["weight_semantic_class"], 0.02, (0.5, 1.5, 0.8))
    p, lt, loss_out = L.fused_forward(m, t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, intr, targets,
                                      True)
    L.fused_backward(m, p, lt, loss_out, scale, True, upstream=ups)
    torch.cuda.synchronize()
    got = [g.clone() for g in L._voxel_grads(m, p, n)]

    # the items this test is about were rendered and registered
    imgs = [x[:I] for x in (m.image_color, m.image_depth, m.image_normal, m.image_semantic)]
    hit = imgs[1] != NINF
    sem_hit = imgs[3][hit]
    assert bool(torch.isnan(sem_hit).any()) and bool((sem_hit[:, 0] == NINF).any())
    assert bool(torch.isinf(sem_hit[:, 1:]).any()) and bool((imgs[0][hit] == NINF).any())

    # per-pixel route: gradient images of the same loss (same normalisers, same scale), then the plain gather
    px = I * m.height * m.width
    g_col, g_dep, g_sem = (torch.empty_like(x) for x in (imgs[0], imgs[1], imgs[3]))
    N.check(N.lib.spsg_losses2d_backward(ctypes.byref(lt), N.ptr(imgs[0]), N.ptr(imgs[1]), N.ptr(imgs[3]), px,
                                         N.ptr(loss_out), N.ptr(scale), N.ptr(g_col), N.ptr(g_dep), N.ptr(g_sem),
                                         rc._stream(dev)))
    if upstream:
        g_col, g_sem = g_col + ups[0], g_sem + ups[3]
    dims = m.dims3d
    rc.backward(g_col, g_dep, torch.zeros_like(imgs[2]), g_sem, m.sparse_mapping, m.mapping3dto2d, m.mapping3dto2d_num,
                [m.batch_size, dims[2], dims[1], dims[0], n], m.d_color, m.d_depth, m.d_normal, m.d_semantic,
                views_per_chunk=F, grads_cleared=False, workspace_owner=m.workspace, flags=m.flags)
    torch.cuda.synchronize()
    want = [g.clone() for g in L._voxel_grads(m, p, n)]
    for name, a, b in zip(("sdf", "color", "normal", "semantic"), got, want):
        assert _same(a, b), "%s: %d entries differ from the per-pixel route" % (name, int((a != b).sum()))
    assert bool(torch.isnan(got[3]).any()), "no NaN logits reached a voxel gradient"
