"""All-pixels mode (SPSG_FLAG_ALL_PIXELS, ``RaycastRGBD(..., max_pixels_per_voxel=None)``): voxel gradients that average
every pixel a (voxel, view) received, without the voxel -> pixel table.  Exact gradients against an oracle built from the
renderings, agreement with the table mode where nothing overflows, schedule independence, the entry-point routes, the
memory it saves, autograd and a bit-reproducible training step.  Helpers: tests/fuzz_all_pixels.py."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from spsg_b200 import _native as N
from spsg_b200 import synthetic as S
from tests import fuzz_all_pixels as A
from tests import fuzz_deterministic as D

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ALL, DET = N.SPSG_FLAG_ALL_PIXELS, N.SPSG_FLAG_DETERMINISTIC


def finite(x):
    return torch.where(torch.isfinite(x), x, torch.zeros_like(x))


def setup(dev, B, F, w, h, seed, close=1.0, zoom=1.0, per_view=False):
    t, n, batch = D.room(dev, B, seed, view_payload=F if per_view else 0)
    view, intr = A.cameras(B * F, np.random.default_rng(seed), w, h, close, zoom)
    return t, n, batch, torch.from_numpy(view).to(dev), torch.from_numpy(intr).to(dev)


# B, F, (W, H), per-view normals, zoom: close cameras, most rows over 64 pixels.  B = 1 renders with 24-warp CTAs and B = 8
# at 320x256 with 28-warp CTAs; zoom 8 puts rows above the shared-memory sort's 4096 entries
EXACT_CASES = [(1, 1, (320, 256), False, 8.0), (3, 3, (160, 128), False, 2.0), (8, 1, (320, 256), False, 1.0),
               (3, 3, (320, 256), True, 2.0), (1, 3, (320, 256), True, 8.0), (8, 3, (160, 128), False, 2.0)]


@pytest.mark.parametrize("B,F,wh,per_view,zoom", EXACT_CASES)
def test_exact_gradients_and_schedules(cuda_device, B, F, wh, per_view, zoom):
    hit, over, longest = A.check_case(cuda_device, B, F, wh[0], wh[1], 1.0, "plain", seed=B * 10 + F, flags=DET,
                                      per_view=per_view, zoom=zoom, what="B=%d F=%d" % (B, F))
    print("rows hit %d, over 64: %d, largest %d" % (hit, over, longest))
    assert over > 0, (hit, over)
    if zoom == 8.0:
        assert longest > A.SMEM_SORT, longest


@pytest.mark.parametrize("variant", ["fused", "fused_up"])
@pytest.mark.parametrize("F,zoom", [(1, 4.0), (3, 1.0)])
def test_fused_gradients_and_schedules(cuda_device, variant, F, zoom):
    hit, over, longest = A.check_case(cuda_device, 2, F, 160, 128, 1.0, variant, seed=F + 3, flags=DET, zoom=zoom,
                                      what="%s F=%d" % (variant, F))
    assert over > 0


@pytest.mark.parametrize("variant", ["plain", "fused_up"])
def test_default_mode_against_the_float64_gather(cuda_device, variant):
    A.check_case(cuda_device, 3, 2, 160, 128, 1.0, variant, seed=21, zoom=2.0, schedules=(0,), what=variant)


@pytest.mark.parametrize("variant", ["plain", "fused", "fused_up"])
@pytest.mark.parametrize("det", [False, True])
def test_table_mode_agrees_where_nothing_overflows(cuda_device, variant, det):
    """Far cameras at 160x128: no row reaches 64 pixels.  Renderings, counts and loss_out are the table mode's bit for bit;
    under DETERMINISTIC the gradients too."""
    B, F, w, h = 3, 2, 160, 128
    t, n, batch, view, intr = setup(cuda_device, B, F, w, h, seed=31, close=0.0)
    out = []
    for mode in (0, ALL):
        flags = mode | (DET if det else 0)
        m = D.raycaster(cuda_device, B, F, w, h, n, None if mode else 64, flags)
        im, _, num, loss_out, grads, _ = D.run_once(m, t, view, intr, variant, seed=31)
        out.append((im, num[:F * n], loss_out, grads))
    (ia, na, la, ga), (ib, nb, lb, gb) = out
    assert 0 < na.max() <= 64
    for a, b in zip(ia, ib):
        assert np.array_equal(D.bits(a), D.bits(b))
    assert np.array_equal(na, nb)
    if det:
        assert la is None or np.array_equal(D.bits(la), D.bits(lb))
        assert np.array_equal(D.bits(ga), D.bits(gb))
    else:  # (the default mode's float atomics: each mode's own runs differ in the last bits)
        assert la is None or np.allclose(la, lb, rtol=1e-6, atol=0)
        np.testing.assert_allclose(ga, gb, rtol=1e-5, atol=1e-6 * float(np.abs(gb).max()))


def test_counts_and_losses_match_the_table_mode_when_rows_overflow(cuda_device):
    B, F, w, h = 2, 2, 160, 128
    t, n, batch, view, intr = setup(cuda_device, B, F, w, h, seed=33, zoom=2.0)
    out = []
    for P in (64, None):
        m = D.raycaster(cuda_device, B, F, w, h, n, P, DET | (ALL if P is None else 0))
        im, _, num, loss_out, _, _ = D.run_once(m, t, view, intr, "fused", seed=33)
        out.append((im, num[:F * n], loss_out))
    assert (out[0][1] > 64).any()
    for a, b in zip(out[0][0], out[1][0]):
        assert np.array_equal(D.bits(a), D.bits(b))
    assert np.array_equal(out[0][1], out[1][1])
    assert np.array_equal(D.bits(out[0][2]), D.bits(out[1][2]))


def _grads(leaves):
    return [x.grad.clone() for x in leaves]


def test_packed_locs_prebuilt_index_and_retain_graph(cuda_device):
    from spsg_b200 import raycast_rgbd_cuda as rc
    from spsg_b200 import sparsify
    B, F, w, h = 2, 2, 160, 128
    t, n, batch, view, intr = setup(cuda_device, B, F, w, h, seed=4, zoom=2.0)
    keys = ("sdf", "color", "normal", "semantic")
    g = torch.Generator(device="cpu").manual_seed(4)
    ups = None
    res = []
    for route in ("int64", "packed"):
        m = D.raycaster(cuda_device, B, F, w, h, n, None, ALL | DET)
        locs = t["locs"] if route == "int64" else rc.pack_locs_host(torch.from_numpy(batch["locs"]), B, S.DIMS_ZYX).to(cuda_device)
        leaves = [t[k].clone().requires_grad_(True) for k in keys]
        outs = m(locs, *leaves, view, intr)
        if ups is None:
            ups = [torch.randn(o.shape, generator=g).to(cuda_device) for o in outs]
        torch.autograd.backward(outs, ups, retain_graph=True)
        first = _grads(leaves)
        torch.autograd.backward(outs, ups)  # second backward over the retained graph: rebuilds the segments, adds g again
        for a, x in zip(first, leaves):
            assert torch.equal(x.grad, 2 * a)
        res.append(first)
    for a, b in zip(*res):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))

    # index + brick written by the compaction: the module's next forward takes SPSG_FLAG_INDEX_PREBUILT
    sdf = torch.stack([torch.from_numpy(S.sdf_volume(s)[0]) for s in range(4, 4 + B)])[:, None].contiguous().to(cuda_device)
    col = torch.rand((B, 3) + tuple(S.DIMS_ZYX), generator=g).to(cuda_device)
    n2 = int((sdf.abs() < S.TRUNCATION).sum())
    grads = []
    for prebuilt in (True, False):
        m2 = D.raycaster(cuda_device, B, F, w, h, n2, None, ALL | DET)
        locs, v_sdf, v_col = sparsify.sparsify_predictions(sdf, S.TRUNCATION, None, col, raycaster=m2 if prebuilt else None)
        nrm = torch.from_numpy(D.O.voxel_normals(n2)).to(cuda_device)
        sem = torch.randn(n2, 14, generator=torch.Generator(device="cpu").manual_seed(5)).to(cuda_device)
        flags_seen = []
        real = N.lib.spsg_raycast_forward_indexed

        def spy(p, *args):
            flags_seen.append(p._obj.flags)
            return real(p, *args)
        N.lib.spsg_raycast_forward_indexed = spy
        try:
            leaves = [x.clone().requires_grad_(True) for x in (v_sdf, v_col, nrm, sem)]
            outs = m2(locs, *leaves, view, intr)
        finally:
            N.lib.spsg_raycast_forward_indexed = real
        assert bool(flags_seen[0] & N.SPSG_FLAG_INDEX_PREBUILT) == prebuilt and flags_seen[0] & ALL
        finite(outs[1]).sum().backward()
        grads.append(_grads(leaves))
    for a, b in zip(*grads):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))


def test_grads_cleared_on_and_off(cuda_device):
    """render_loss_and_voxel_grads lets the forward clear the gradient rows; a backward without that clears them itself."""
    from spsg_b200 import losses as L
    B, F, w, h = 2, 3, 160, 128
    t, n, batch, view, intr = setup(cuda_device, B, F, w, h, seed=6, zoom=2.0)
    depth_t, color_t, label_t, cw = D.targets(B * F, w, h, cuda_device, np.random.default_rng(6))
    m = D.raycaster(cuda_device, B, F, w, h, n, None, ALL | DET)
    _, grads = L.render_loss_and_voxel_grads(m, t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, intr,
                                             images_depth=depth_t, images_color=color_t, target2d_label=label_t,
                                             weight_semantic_class=cw)
    cleared = [x.clone() for x in grads]
    targets = (depth_t, color_t, None, label_t, cw, 0.02, (1.0, 1.0, 1.0))
    p, tg, loss_out = L.fused_forward(m, t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, intr, targets,
                                      False)
    for x in (m.d_color, m.d_depth, m.d_normal, m.d_semantic):
        x.fill_(7.0)  # stale rows: the backward must overwrite every one of [0, N)
    L.fused_backward(m, p, tg, loss_out, torch.ones((), device=cuda_device), False)
    for a, b in zip(cleared, L._voxel_grads(m, p, n)):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))


def test_module_without_a_table_allocates_none(cuda_device):
    """At the training step's shape (B = 8, F = 1, 640000 rows per chunk, 320x256) the table is 1.31 GB."""
    from spsg_b200.raycast_rgbd import RaycastRGBD
    torch.cuda.synchronize()
    sizes = {}
    for P in (64, None):
        torch.cuda.empty_cache()
        before = torch.cuda.memory_allocated(cuda_device)
        m = RaycastRGBD(8, S.DIMS_ZYX, 320, 256, 5.0, 300.0, S.THRESH_SAMPLE_DIST, S.RAY_INCREMENT,
                        max_num_locs_per_sample=640000, max_pixels_per_voxel=P, device=cuda_device)
        sizes[P] = torch.cuda.memory_allocated(cuda_device) - before
        assert bool(m.flags & ALL) == (P is None)
        if P is None:
            assert m.mapping3dto2d.numel() == 0
        del m
    saved = sizes[64] - sizes[None]
    print("table memory saved at the train-step shape: %d bytes" % saved)
    assert saved >= 8 * 640000 * 64 * 4


def test_backward_in_the_other_mode_raises(cuda_device):
    from spsg_b200 import raycast_rgbd_cuda as rc
    B, F, w, h = 1, 1, 88, 60
    t, n, batch, view, intr = setup(cuda_device, B, F, w, h, seed=12)
    for P in (None, 64):
        m = D.raycaster(cuda_device, B, F, w, h, n, P, ALL if P is None else 0)
        m(t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, intr)
        g = [torch.ones_like(x) for x in (m.image_color, m.image_depth, m.image_normal, m.image_semantic)]
        table = m.mapping3dto2d if P else torch.zeros(n, 64, dtype=torch.int32, device=cuda_device)
        other = 0 if P is None else ALL
        with pytest.raises(RuntimeError, match="matching forward"):
            rc.backward(*g, m.sparse_mapping, table, m.mapping3dto2d_num, [B, 64, 64, 128, n], m.d_color, m.d_depth,
                        m.d_normal, m.d_semantic, workspace_owner=m.workspace, flags=other)
        # the same call in the forward's own mode runs
        rc.backward(*g, m.sparse_mapping, m.mapping3dto2d, m.mapping3dto2d_num, [B, 64, 64, 128, n], m.d_color,
                    m.d_depth, m.d_normal, m.d_semantic, workspace_owner=m.workspace, flags=m.flags)


_TRAIN_SCRIPT = r"""
import json, sys
import torch
sys.path.insert(0, %(root)r)
torch.backends.cudnn.benchmark = False
torch.use_deterministic_algorithms(True)
from spsg_b200 import _native as N
from spsg_b200 import synthetic as S
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
    step = _step(dev, model, max_pixels_per_voxel=None)
    step.raycaster.flags |= sched
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    loss = step(dict(sample), optimizer=opt)
    torch.cuda.synchronize()
    num = step.raycaster.mapping3dto2d_num[:step.last["num_locs"]]
    res.append(dict(loss=float(loss), bits=torch.cat([p.detach().reshape(-1) for p in model.parameters()]).view(torch.int32).tolist(),
                    rows=int((num > 0).sum()), over=int((num > 64).sum()), table=step.raycaster.mapping3dto2d.numel()))
a, b = res
print(json.dumps(dict(loss=[a["loss"], b["loss"]], same_loss=a["loss"] == b["loss"], rows=a["rows"], over=a["over"],
                      table=a["table"], differing_params=sum(x != y for x, y in zip(a["bits"], b["bits"])),
                      params=len(a["bits"]))))
"""


def test_train_step_without_a_table_is_bit_reproducible(cuda_device):
    env = dict(os.environ, CUBLAS_WORKSPACE_CONFIG=":4096:8")
    out = subprocess.run([sys.executable, "-c", _TRAIN_SCRIPT % dict(root=ROOT)], cwd=ROOT, env=env, capture_output=True,
                         text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-4000:]
    r = json.loads(out.stdout.strip().splitlines()[-1])
    print("all-pixels deterministic train step:", r)
    assert r["table"] == 0 and r["over"] > 0, r
    assert r["same_loss"] and r["differing_params"] == 0, r


def test_fuzz_slice(cuda_device):
    assert A.run(cases=8, seed0=5, dev=cuda_device) == 0
