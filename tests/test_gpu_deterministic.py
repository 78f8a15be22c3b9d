"""Deterministic mode (SPSG_FLAG_DETERMINISTIC, or torch.use_deterministic_algorithms(True)): canonical voxel -> pixel
tables against the renderings, schedule independence of tables, losses and gradients, exact plain gradients, the Python
switch, and a bit-reproducible training step.  Helpers: tests/fuzz_deterministic.py."""
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from spsg_b200 import _native as N
from spsg_b200 import synthetic as S
from tests import fuzz_deterministic as D

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def finite(x):
    return torch.where(torch.isfinite(x), x, torch.zeros_like(x))


@pytest.fixture
def torch_deterministic():
    before = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(before)


# B, F, max_pixels_per_voxel, (W, H), per-view normals: P in {1, 7, 64}, F in {1, 2, 3}, B in {1, 3, 8}; B = 1 renders with
# 24-warp CTAs and shared-memory maps by default, B = 8 at 320x256 with 28-warp CTAs and L1 maps (the schedule flags
# force the other map path in every case)
TABLE_CASES = [(1, 1, 64, (320, 256), False), (1, 2, 7, (320, 256), False), (3, 3, 1, (160, 128), False),
               (8, 1, 64, (320, 256), False), (3, 2, 64, (320, 256), True), (8, 3, 7, (160, 128), False),
               (3, 3, 64, (320, 256), True)]


@pytest.mark.parametrize("B,F,P,wh,per_view", TABLE_CASES)
def test_tables_schedules_and_exact_gradients(cuda_device, B, F, P, wh, per_view):
    hit, over = D.check_case(cuda_device, B, F, P, wh[0], wh[1], 1.0, "plain", seed=B * 10 + F, per_view=per_view,
                             what="B=%d F=%d P=%d" % (B, F, P))
    assert over > 0, (hit, over)


@pytest.mark.parametrize("variant", ["fused", "fused_up"])
@pytest.mark.parametrize("F", [1, 3])
def test_fused_schedule_independence(cuda_device, variant, F):
    D.check_case(cuda_device, 2, F, 64, 160, 128, 0.7, variant, seed=F + 3, what="%s F=%d" % (variant, F))


def _tables_of(m, view, batch, F, P):
    images = view.shape[0]
    vox = D.voxel_of_pixels(m.image_depth[:images].detach().cpu().numpy(), m.image_normal[:images].detach().cpu().numpy())
    c = D.canonical_tables(vox, batch["locs"][:, 3], F, P)
    return D.check_tables(c, m.mapping3dto2d.cpu().numpy(), m.mapping3dto2d_num.cpu().numpy())


def test_packed_locs_and_prebuilt_index_routes(cuda_device):
    from spsg_b200 import raycast_rgbd_cuda as rc
    from spsg_b200 import sparsify
    B, F, P, w, h = 2, 2, 64, 160, 128
    t, n, batch = D.room(cuda_device, B, seed=4)
    view, intr = D.cameras(B * F, np.random.default_rng(4), w, h)
    view, intr = torch.from_numpy(view).to(cuda_device), torch.from_numpy(intr).to(cuda_device)
    m = D.raycaster(cuda_device, B, F, w, h, n, P, N.SPSG_FLAG_DETERMINISTIC)
    packed = rc.pack_locs_host(torch.from_numpy(batch["locs"]), B, S.DIMS_ZYX).to(cuda_device)
    m(packed, t["sdf"], t["color"], t["normal"], t["semantic"], view, intr)
    assert _tables_of(m, view, batch, F, P)[1] > 0

    # index + brick written by the compaction (SPSG_FLAG_INDEX_PREBUILT on the module's next forward)
    sdf = torch.stack([torch.from_numpy(S.sdf_volume(s)[0]) for s in range(4, 4 + B)])[:, None].contiguous().to(cuda_device)
    g = torch.Generator(device="cpu").manual_seed(5)
    col = torch.rand((B, 3) + tuple(S.DIMS_ZYX), generator=g).to(cuda_device)
    m2 = D.raycaster(cuda_device, B, F, w, h, int((sdf.abs() < S.TRUNCATION).sum()), P, N.SPSG_FLAG_DETERMINISTIC)
    locs, v_sdf, v_col = sparsify.sparsify_predictions(sdf, S.TRUNCATION, None, col, raycaster=m2)
    n2 = locs.shape[0]
    nrm = torch.from_numpy(D.O.voxel_normals(n2)).to(cuda_device)
    sem = torch.randn(n2, 14, generator=g).to(cuda_device)
    flags_seen = []
    real = N.lib.spsg_raycast_forward_indexed

    def spy(p, *args):
        flags_seen.append(p._obj.flags)
        return real(p, *args)
    N.lib.spsg_raycast_forward_indexed = spy
    try:
        m2(locs, v_sdf, v_col, nrm, sem, view, intr)
    finally:
        N.lib.spsg_raycast_forward_indexed = real
    assert flags_seen and flags_seen[0] & N.SPSG_FLAG_INDEX_PREBUILT and flags_seen[0] & N.SPSG_FLAG_DETERMINISTIC
    assert _tables_of(m2, view, {"locs": locs.cpu().numpy()}, F, P)[1] > 0


@pytest.mark.parametrize("B,F,P", [(1, 1, 64), (3, 2, 7)])
def test_flag_off_and_on_agree(cuda_device, B, F, P):
    """Renderings and counts bit-identical; table entries the same sets wherever nothing overflowed."""
    w, h = 160, 128
    t, n, batch = D.room(cuda_device, B, seed=7)
    view, intr = D.cameras(B * F, np.random.default_rng(7), w, h, close=0.5)
    view, intr = torch.from_numpy(view).to(cuda_device), torch.from_numpy(intr).to(cuda_device)
    out = []
    for flags in (0, N.SPSG_FLAG_DETERMINISTIC):
        m = D.raycaster(cuda_device, B, F, w, h, n, P, flags)
        imgs = m(t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, intr)
        out.append(([x.clone() for x in imgs], m.mapping3dto2d[:F * n].clone(), m.mapping3dto2d_num[:F * n].clone()))
    (ia, ma, na), (ib, mb, nb) = out
    for a, b in zip(ia, ib):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))
    assert torch.equal(na, nb)
    ok = (na > 0) & (na <= P)
    used = torch.arange(P, device=cuda_device)[None, :] < na[:, None]
    fill = torch.iinfo(torch.int32).max
    sa = torch.where(used, ma, fill)[ok].sort(1).values
    sb = torch.where(used, mb, fill)[ok].sort(1).values
    assert torch.equal(sa, sb)
    assert torch.equal(sb, torch.where(used, mb, fill)[ok])  # deterministic rows are already ascending


def test_loss_values_match_reference(cuda_device, torch_deterministic):
    from oracle import losses_ref as R
    from spsg_b200.losses import losses_2d, render_with_2d_losses
    B, F, w, h = 2, 2, 160, 128
    t, n, batch = D.room(cuda_device, B, seed=9)
    view, intr = D.cameras(B * F, np.random.default_rng(9), w, h, close=0.5)
    view, intr = torch.from_numpy(view).to(cuda_device), torch.from_numpy(intr).to(cuda_device)
    depth_t, color_t, label_t, cw = D.targets(B * F, w, h, cuda_device, np.random.default_rng(9))
    m = D.raycaster(cuda_device, B, F, w, h, n, 64, 0)
    total, terms, imgs = render_with_2d_losses(m, t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, intr,
                                               images_depth=depth_t, images_color=color_t, target2d_label=label_t,
                                               weight_semantic_class=cw, voxelsize=S.VOXELSIZE)
    r_color, r_depth, _, r_sem = (x.clone() for x in imgs)
    torch.use_deterministic_algorithms(False)  # (the reference expressions are not the subject here)
    want = torch.stack([R.depth_l1_loss(r_depth, depth_t[:, None], S.VOXELSIZE), R.compute_2dcolor_loss(r_color, color_t, None),
                        R.semantic_2d_ce_loss(r_sem, label_t[..., None], cw)])
    torch.use_deterministic_algorithms(True)
    torch.testing.assert_close(terms, want, rtol=1e-5, atol=1e-7)
    torch.testing.assert_close(total, want.sum(), rtol=1e-5, atol=1e-7)
    total2, terms2 = losses_2d(r_color, r_depth, r_sem, images_depth=depth_t, images_color=color_t,
                               target2d_label=label_t, weight_semantic_class=cw, voxelsize=S.VOXELSIZE)
    torch.testing.assert_close(terms2, want, rtol=1e-5, atol=1e-7)
    torch.testing.assert_close(total2, want.sum(), rtol=1e-5, atol=1e-7)


def test_standalone_losses_do_not_depend_on_the_grid(cuda_device):
    """spsg_losses2d_forward_deterministic: the loss block of two calls is bit-identical (the scratch size does not enter),
    and equal to the default op's to 1e-5."""
    from spsg_b200.losses import _targets_struct
    g = torch.Generator(device="cpu").manual_seed(3)
    P = 300001
    col = torch.rand(P, 3, generator=g).to(cuda_device)
    dep = (torch.rand(P, generator=g) * 50).to(cuda_device)
    sem = (torch.randn(P, 14, generator=g) * 4).to(cuda_device)
    td = torch.rand(P, generator=g).to(cuda_device)
    tc = torch.rand(P, 3, generator=g).to(cuda_device)
    lab = torch.randint(0, 15, (P,), generator=g, dtype=torch.uint8).to(cuda_device)
    st = torch.cuda.current_stream(cuda_device).cuda_stream

    def run(fn, k):
        tg = _targets_struct(1, 1, P, td, tc, None, lab, None, 0.02, (1.0, 0.5, 0.25))
        out = torch.empty(8, device=cuda_device)
        scratch = torch.empty(N.lib.spsg_losses2d_deterministic_scratch_bytes(P) + k, dtype=torch.uint8, device=cuda_device)
        N.check(fn(ctypes.byref(tg), N.ptr(col), N.ptr(dep), N.ptr(sem), P, N.ptr(out), N.ptr(scratch), scratch.numel(), st))
        return out
    a = run(N.lib.spsg_losses2d_forward_deterministic, 0)
    b = run(N.lib.spsg_losses2d_forward_deterministic, 4096)
    assert torch.equal(a.view(torch.int32), b.view(torch.int32))
    c = run(N.lib.spsg_losses2d_forward, 0)
    torch.testing.assert_close(a[:7], c[:7], rtol=1e-5, atol=0)


def test_python_switch_reaches_every_entry_point(cuda_device, torch_deterministic):
    from spsg_b200 import losses as L
    from spsg_b200 import raycast_rgbd_cuda as rc
    B, F, P, w, h = 2, 1, 16, 160, 128
    t, n, batch = D.room(cuda_device, B, seed=11)
    view, intr = D.cameras(B * F, np.random.default_rng(11), w, h)
    view, intr = torch.from_numpy(view).to(cuda_device), torch.from_numpy(intr).to(cuda_device)
    depth_t, color_t, label_t, cw = D.targets(B * F, w, h, cuda_device, np.random.default_rng(11))

    # RaycastRGBD with flags 0
    m = D.raycaster(cuda_device, B, F, w, h, n, P, 0)
    sdf = t["sdf"].clone().requires_grad_(True)
    imgs = m(t["locs"], sdf, t["color"], t["normal"], t["semantic"], view, intr)
    assert _tables_of(m, view, batch, F, P)[1] > 0
    finite(imgs[1]).sum().backward()
    # render_with_2d_losses
    m = D.raycaster(cuda_device, B, F, w, h, n, P, 0)
    total, _, _ = L.render_with_2d_losses(m, t["locs"], sdf, t["color"], t["normal"], t["semantic"], view, intr,
                                          images_depth=depth_t, target2d_label=label_t, weight_semantic_class=cw)
    assert _tables_of(m, view, batch, F, P)[1] > 0
    total.backward()
    # render_loss_and_voxel_grads
    m = D.raycaster(cuda_device, B, F, w, h, n, P, 0)
    L.render_loss_and_voxel_grads(m, t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, intr,
                                  images_depth=depth_t, images_color=color_t)
    assert _tables_of(m, view, batch, F, P)[1] > 0
    # the drop-in extension module with bare tensors, as the reference's wrapper calls it
    m = D.raycaster(cuda_device, B, F, w, h, n, P, 0)
    sm = torch.empty_like(m.sparse_mapping)
    opts = [w, h, 0.0, 300.0, S.THRESH_SAMPLE_DIST, S.RAY_INCREMENT, S.DIMS_ZYX[2], S.DIMS_ZYX[1], S.DIMS_ZYX[0]]
    rc.construct_dense_sparse_mapping(t["locs"], sm)
    rc.forward(sm, t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, m.image_color, m.image_depth,
               m.image_normal, m.image_semantic, m.mapping3dto2d, m.mapping3dto2d_num, intr, opts)
    assert _tables_of(m, view, batch, F, P)[1] > 0
    g = [torch.ones_like(x) for x in (m.image_color, m.image_depth, m.image_normal, m.image_semantic)]
    rc.backward(*g, sm, m.mapping3dto2d, m.mapping3dto2d_num, [B, 64, 64, 128, n], m.d_color, m.d_depth, m.d_normal,
                m.d_semantic)
    # ... and the same backward with the switch off is a backward in the other mode
    torch.use_deterministic_algorithms(False)
    with pytest.raises(RuntimeError, match="matching forward"):
        rc.backward(*g, sm, m.mapping3dto2d, m.mapping3dto2d_num, [B, 64, 64, 128, n], m.d_color, m.d_depth, m.d_normal,
                    m.d_semantic)
    torch.use_deterministic_algorithms(True)


@pytest.mark.parametrize("path", ["module", "fused"])
def test_backward_in_the_other_mode_raises(cuda_device, path):
    from spsg_b200 import losses as L
    B, F, w, h = 1, 1, 88, 60
    t, n, batch = D.room(cuda_device, B, seed=12)
    view, intr = D.cameras(B * F, np.random.default_rng(12), w, h)
    view, intr = torch.from_numpy(view).to(cuda_device), torch.from_numpy(intr).to(cuda_device)
    before = torch.are_deterministic_algorithms_enabled()
    try:
        for fwd_mode in (True, False):
            m = D.raycaster(cuda_device, B, F, w, h, n, 64, 0)
            sdf = t["sdf"].clone().requires_grad_(True)
            torch.use_deterministic_algorithms(fwd_mode)
            if path == "module":
                out = finite(m(t["locs"], sdf, t["color"], t["normal"], t["semantic"], view, intr)[1]).sum()
            else:
                depth_t = torch.ones(B * F, h, w, device=cuda_device)
                out = L.render_with_2d_losses(m, t["locs"], sdf, t["color"], t["normal"], t["semantic"], view, intr,
                                              images_depth=depth_t)[0]
            torch.use_deterministic_algorithms(not fwd_mode)
            with pytest.raises(RuntimeError, match="matching forward"):
                out.backward()
    finally:
        torch.use_deterministic_algorithms(before)


_TRAIN_SCRIPT = r"""
import json, sys
import torch
sys.path.insert(0, %(root)r)
torch.backends.cudnn.benchmark = False
torch.use_deterministic_algorithms(%(det)s)
from spsg_b200 import _native as N
from spsg_b200 import synthetic as S
from spsg_b200 import train_step
from tests.test_gpu_head_formats import DIMS, W, H, _Generator, _step
dev = torch.device("cuda", 0)
torch.manual_seed(1234)
base = _Generator().to(dev)
sample = S.make_train_sample([0, 1], 1, dims_zyx=DIMS, width=W, height=H,
                             view_kw=dict(center=(16.0, 16.0, 11.0), radius=5.0, height=15.0))
sample = {k: torch.from_numpy(v).to(dev) for k, v in sample.items()}
sample["known"] = None
res = []
for sched in (0, N.SPSG_FLAG_GLOBAL_MAPS | N.SPSG_FLAG_NO_BRICK_SKIP):
    model = _Generator().to(dev)
    model.load_state_dict(base.state_dict())
    step = _step(dev, model)
    step.raycaster.flags |= sched
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    loss = step(dict(sample), optimizer=opt)
    torch.cuda.synchronize()
    num = step.raycaster.mapping3dto2d_num[:step.last["num_locs"]]
    res.append(dict(loss=float(loss), bits=torch.cat([p.detach().reshape(-1) for p in model.parameters()]).view(torch.int32).tolist(),
                    rows=int((num > 0).sum()), over=int((num > step.raycaster.mapping3dto2d.shape[1]).sum())))
a, b = res
print(json.dumps(dict(loss=[a["loss"], b["loss"]], same_loss=a["loss"] == b["loss"], rows=a["rows"], over=a["over"],
                      differing_params=sum(x != y for x, y in zip(a["bits"], b["bits"])), params=len(a["bits"]))))
"""


def train_step_pair(det):
    """Two Adam steps from the same generator state, the second raycaster on another schedule, in a fresh process."""
    env = dict(os.environ, CUBLAS_WORKSPACE_CONFIG=":4096:8")
    out = subprocess.run([sys.executable, "-c", _TRAIN_SCRIPT % dict(root=ROOT, det=bool(det))], cwd=ROOT, env=env,
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-4000:]
    return json.loads(out.stdout.strip().splitlines()[-1])


def test_train_step_is_bit_reproducible(cuda_device):
    r = train_step_pair(True)
    print("deterministic train step:", r)
    assert r["over"] > 0, r
    assert r["same_loss"] and r["differing_params"] == 0, r


def test_fuzz_slice(cuda_device):
    assert D.run(cases=10, seed0=5, dev=cuda_device) == 0
