"""Configurable semantic class count C (``RaycastRGBD(..., num_classes=C)``, spsg_raycast_params.semantic_channels).

Geometry does not depend on C, so a C-class render is checked against the 14-class render of the same voxels: colour,
depth, normal, mapping3dto2d_num and (deterministic) tables bit for bit, and every semantic pixel is its hit voxel's
row (the voxel id rides in the normal payload, tests/gather_oracle.py).  Gradients: per channel, the C-generic gather adds
exactly what the 14-channel gather adds, so under SPSG_FLAG_DETERMINISTIC a C-channel backward equals, bit for bit, 14-channel
backwards of the same images cut into 14-channel windows.  Losses against the literal PyTorch expressions.
Helpers shared with tests/fuzz_semantic_classes.py."""
import pytest
import torch

from spsg_b200 import _native as N
from spsg_b200 import losses
from spsg_b200 import synthetic as S
from spsg_b200.raycast_rgbd import RaycastRGBD
from tests import fuzz_semantic_classes as Z

pytestmark = pytest.mark.gpu

DET, GEN = N.SPSG_FLAG_DETERMINISTIC, N.SPSG_FLAG_GENERIC_SEMANTIC


def bits(t):
    return t.detach().contiguous().view(torch.int32)


@pytest.mark.parametrize("C", [1, 2, 13, 15, 16, 17, 20, 32, 41, 64])
@pytest.mark.parametrize("B", [1, 3, 8])
@pytest.mark.parametrize("F", [1, 3])
def test_geometry_equals_the_14_class_render(cuda_device, C, B, F):
    Z.check_render(cuda_device, C, B, F, 160, 128, seed=C + 7 * B + F, flags=DET)


@pytest.mark.parametrize("C", [20, 64])
@pytest.mark.parametrize("flags", [DET, 0])
def test_geometry_at_c3_size(cuda_device, C, flags):
    """8 chunks x 5 views at 320x256: enough tiles for the 28-warp forward CTAs."""
    Z.check_render(cuda_device, C, 8, 5, 320, 256, seed=C, flags=flags)


@pytest.mark.parametrize("extra", [0, DET, DET | N.SPSG_FLAG_ALL_PIXELS, DET | N.SPSG_FLAG_GLOBAL_MAPS,
                                   DET | N.SPSG_FLAG_SMEM_MAPS, N.SPSG_FLAG_DETERMINISTIC_GRADS | DET])
@pytest.mark.parametrize("F,per_view", [(1, False), (3, False), (3, True)])
def test_generic_path_at_14_is_bit_identical(cuda_device, extra, F, per_view):
    """SPSG_FLAG_GENERIC_SEMANTIC at C = 14 against the specialised kernels: renderings, tables, loss_out and the
    gradients of the plain, fused and fused + upstream backwards (the default mode's fused forward epilogue included)."""
    _compare_generic(cuda_device, extra, 3, F, 160, 128, per_view)


@pytest.mark.parametrize("extra", [DET, 0])
def test_generic_path_at_14_at_c3_size(cuda_device, extra):
    """The same with the 28-warp forward CTAs (8 chunks x 5 views at 320x256)."""
    _compare_generic(cuda_device, extra, 8, 5, 320, 256, False)


def _compare_generic(dev, extra, B, F, w, h, per_view):
    det = bool(extra & DET)
    # default mode: which 64 pixels an overflowing row keeps, and the order of the loss and several-view atomics, depend
    # on the schedule: far cameras (no row over 64 pixels), and the sums within 1e-5
    runs = [Z.run_all_routes(dev, 14, B, F, w, h, seed=F + 11, flags=extra | g, per_view=per_view,
                             close=1.0 if det else 0.0) for g in (0, GEN)]
    for key in runs[0]:
        a, b = runs[0][key], runs[1][key]
        if det or not key.startswith(("grad_", "loss")):
            assert torch.equal(bits(a), bits(b)), key
        else:
            assert torch.allclose(a, b, rtol=1e-5, atol=1e-6), key


@pytest.mark.parametrize("C", [1, 2, 13, 20, 41, 64])
@pytest.mark.parametrize("F,flags", [(1, DET), (3, DET), (3, DET | N.SPSG_FLAG_ALL_PIXELS), (1, DET | N.SPSG_FLAG_GLOBAL_MAPS)])
def test_plain_gradients_equal_14_channel_windows(cuda_device, C, F, flags):
    Z.check_plain_grads(cuda_device, C, 2, F, 160, 128, seed=C + F, flags=flags)


@pytest.mark.parametrize("C", [1, 5, 20, 41, 64])
@pytest.mark.parametrize("weights,ignore", [(False, 0.0), (True, 0.3)])
@pytest.mark.parametrize("terms", [(1.0, 1.0, 1.0), (0.0, 0.0, 1.0), (1.0, 0.5, 0.0)])
def test_losses_against_literal_pytorch(cuda_device, C, weights, ignore, terms):
    Z.check_losses(cuda_device, C, 2, 1, 160, 128, seed=C, weights=weights, ignore=ignore, terms=terms)


@pytest.mark.parametrize("C", [1, 20, 41, 64])
@pytest.mark.parametrize("F", [1, 3])
@pytest.mark.parametrize("upstream", [False, True])
def test_default_mode_fused_path_against_literal_pytorch(cuda_device, C, F, upstream):
    """No SPSG_FLAG_DETERMINISTIC: the fused forward's cross-entropy epilogue, the loss atomics and (F = 3) the gathers
    that add the per-view means with float atomics.  Far cameras: no table row overflows, so the fused and the plain
    backward average the same pixels."""
    Z.check_losses(cuda_device, C, 2, F, 160, 128, seed=C + F, weights=True, ignore=0.2, terms=(1.0, 1.0, 1.0), flags=0,
                   upstream=upstream, close=0.0)


@pytest.mark.parametrize("C", [20, 64])
@pytest.mark.parametrize("F", [1, 3])
def test_default_mode_all_pixels_fused_path_against_literal_pytorch(cuda_device, C, F):
    Z.check_losses(cuda_device, C, 2, F, 160, 128, seed=C + F, weights=True, ignore=0.2, terms=(1.0, 1.0, 1.0),
                   flags=N.SPSG_FLAG_ALL_PIXELS, upstream=True, close=0.5)


@pytest.mark.parametrize("C", [20, 41])
@pytest.mark.parametrize("F", [1, 3])
def test_default_mode_plain_gradients(cuda_device, C, F):
    Z.check_plain_grads(cuda_device, C, 2, F, 160, 128, seed=C + F, flags=0, close=0.0)


@pytest.mark.parametrize("det", [False, True])
def test_losses_deterministic_and_three_views(cuda_device, det):
    torch.use_deterministic_algorithms(det)
    try:
        Z.check_losses(cuda_device, 20, 3, 3, 160, 128, seed=5, weights=True, ignore=0.2, terms=(1.0, 1.0, 1.0))
    finally:
        torch.use_deterministic_algorithms(False)


@pytest.mark.parametrize("C", [1, 3, 14, 20, 41, 64])
def test_label_maps_and_histogram(cuda_device, C):
    g = torch.Generator(device=cuda_device).manual_seed(C)
    sem = torch.rand(2, 33, 47, C, device=cuda_device, generator=g) * 1.5
    sem[0, :5] = -float("inf")          # misses
    sem[1, :3] = 0.0                    # unlabeled
    sem[1, 3, :, 0] = float("nan")      # NaN counts as the maximum
    cat = torch.cat((sem, torch.ones(sem.shape[:-1] + (1,), device=cuda_device)), -1)
    want = torch.max(cat, -1)[1].to(torch.uint8)
    got, hist = losses.labels_from_render(sem, histogram=True)
    assert torch.equal(got, want)
    assert hist.shape == (C + 1,) and torch.equal(hist, torch.bincount(want.flatten().long(), minlength=C + 1))


def test_packed_locs_and_retain_graph(cuda_device):
    Z.check_routes(cuda_device, 20)


@pytest.mark.parametrize("C", [5, 20, 64])
def test_prebuilt_index_from_c_channel_heads(cuda_device, C):
    Z.check_prebuilt(cuda_device, C)


def test_train_step_with_20_classes_against_literal_losses(cuda_device):
    Z.check_train_step(cuda_device, 20)


_TRAIN_SCRIPT = r"""
import json, sys
import torch
sys.path.insert(0, %(root)r)
torch.backends.cudnn.benchmark = False
torch.use_deterministic_algorithms(True)
from spsg_b200 import _native as N
from tests import fuzz_semantic_classes as Z
dev = torch.device("cuda", 0)
torch.manual_seed(1234)
base = Z.GenC(20).to(dev)
sample = Z.train_sample(dev, 20)
res = []
for sched in (0, N.SPSG_FLAG_GLOBAL_MAPS | N.SPSG_FLAG_NO_BRICK_SKIP):
    model = Z.GenC(20).to(dev)
    model.load_state_dict(base.state_dict())
    step = Z.train_step(dev, model, 20, flags=sched)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    loss = step({k: (v.clone() if v is not None else None) for k, v in sample.items()}, optimizer=opt)
    torch.cuda.synchronize()
    res.append(dict(loss=float(loss), n=step.last["num_locs"],
                    bits=torch.cat([p.detach().reshape(-1) for p in model.parameters()]).view(torch.int32).tolist()))
a, b = res
print(json.dumps(dict(loss=[a["loss"], b["loss"]], same_loss=a["loss"] == b["loss"], n=a["n"],
                      differing_params=sum(x != y for x, y in zip(a["bits"], b["bits"])), params=len(a["bits"]))))
"""


def test_train_step_with_20_classes_is_bit_reproducible(cuda_device):
    """Under torch.use_deterministic_algorithms(True), one optimizer step gives the same loss and parameters bit for bit
    with either schedule of the forward (maps through L1 and no block skipping, or the default)."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, CUBLAS_WORKSPACE_CONFIG=":4096:8")
    out = subprocess.run([sys.executable, "-c", _TRAIN_SCRIPT % dict(root=root)], cwd=root, env=env, capture_output=True,
                         text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-4000:]
    r = json.loads(out.stdout.strip().splitlines()[-1])
    print("20-class deterministic train step:", r)
    assert r["n"] > 0 and r["same_loss"] and r["differing_params"] == 0, r


def test_backward_with_another_c_raises(cuda_device):
    from spsg_b200 import raycast_rgbd_cuda as rc
    t, n, batch, view, intr = Z.setup(cuda_device, 1, 1, 80, 64, seed=3)
    m = RaycastRGBD(1, S.DIMS_ZYX, 80, 64, S.DEPTH_MIN, S.DEPTH_MAX, S.THRESH_SAMPLE_DIST, S.RAY_INCREMENT,
                    max_num_locs_per_sample=n, num_classes=20)
    sem = torch.zeros(n, 20, device=cuda_device)
    m(t["locs"], t["sdf"], t["color"], t["normal"], sem, view, intr)
    g = [torch.zeros_like(x) for x in (m.image_color, m.image_depth, m.image_normal)]
    d14 = torch.zeros(n, 14, device=cuda_device)
    with pytest.raises(RuntimeError, match="without a matching forward"):
        rc.backward(g[0], g[1], g[2], torch.zeros(1, 64, 80, 14, device=cuda_device), m.sparse_mapping, m.mapping3dto2d,
                    m.mapping3dto2d_num, [1, S.DIMS_ZYX[2], S.DIMS_ZYX[1], S.DIMS_ZYX[0], n], m.d_color, m.d_depth,
                    m.d_normal, d14, workspace_owner=m.workspace)


def test_out_of_range_c_and_wrong_widths_raise(cuda_device):
    for c in (0, 65):
        with pytest.raises(RuntimeError, match="num_classes"):
            RaycastRGBD(1, S.DIMS_ZYX, 80, 64, S.DEPTH_MIN, S.DEPTH_MAX, S.THRESH_SAMPLE_DIST, S.RAY_INCREMENT,
                        max_num_locs_per_sample=10, num_classes=c)
    t, n, batch, view, intr = Z.setup(cuda_device, 1, 1, 80, 64, seed=3)
    m = RaycastRGBD(1, S.DIMS_ZYX, 80, 64, S.DEPTH_MIN, S.DEPTH_MAX, S.THRESH_SAMPLE_DIST, S.RAY_INCREMENT,
                    max_num_locs_per_sample=n, num_classes=20)
    with pytest.raises(RuntimeError, match="vals_semantics must be"):
        m(t["locs"], t["sdf"], t["color"], t["normal"], torch.zeros(n, 14, device=cuda_device), view, intr)
    with pytest.raises(RuntimeError, match="vals_semantics must be"):
        losses.render_with_2d_losses(m, t["locs"], t["sdf"], t["color"], t["normal"], torch.zeros(n, 21, device=cuda_device),
                                     view, intr, target2d_label=torch.zeros(1, 64, 80, dtype=torch.uint8, device=cuda_device))
    with pytest.raises(RuntimeError, match="class_weight"):
        losses.render_with_2d_losses(m, t["locs"], t["sdf"], t["color"], t["normal"], torch.zeros(n, 20, device=cuda_device),
                                     view, intr, target2d_label=torch.zeros(1, 64, 80, dtype=torch.uint8, device=cuda_device),
                                     weight_semantic_class=torch.ones(14, device=cuda_device))
    with pytest.raises(RuntimeError, match="channels"):
        losses.labels_from_render(torch.zeros(4, 65, device=cuda_device))
    with pytest.raises(RuntimeError, match="class_weight"):
        losses.semantic_2d_ce_loss(torch.zeros(1, 4, 4, 20, device=cuda_device),
                                   torch.zeros(1, 4, 4, dtype=torch.uint8, device=cuda_device), torch.ones(14, device=cuda_device))


def test_fuzz_slice(cuda_device):
    failures = Z.sweep(cuda_device, cases=12, seed=2026)
    assert not failures, failures
