"""Label render (``RaycastRGBD.render_labels``, spsg_raycast_labels), bit for bit:
  * against the one-hot route it replaces (``labels_from_render`` of a forward with the one-hot labels as payload) on every
    route of the forward: one and several chunks, 24- and 28-warp CTAs, debug flags, a grid beyond the shared-memory maps,
    packed and prebuilt index routes, empty chunks and views, N = 0, labels equal to and above C;
  * against the logits route (``labels_from_render(render(logits))``) with NaN, +-inf, ties and maxima at and below 1;
  * module behaviour: no image, table or gradient buffer written, a backward after it raises, module flags ignored;
  * the training step's target labels and the whole step, and the room driver, against their previous routes.
Helpers and the random sweep: tests/fuzz_label_render.py."""
import numpy as np
import pytest
import torch
import torch.nn.functional as Fn

from spsg_b200 import _native as N
from spsg_b200 import losses
from spsg_b200 import raycast_rgbd_cuda as rc
from spsg_b200 import synthetic as S
from tests import fuzz_label_render as L

pytestmark = pytest.mark.gpu

DET, ALL = N.SPSG_FLAG_DETERMINISTIC, N.SPSG_FLAG_ALL_PIXELS


@pytest.mark.parametrize("C", [1, 2, 14, 20, 41, 64])
@pytest.mark.parametrize("B", [1, 3, 8])
@pytest.mark.parametrize("F", [1, 3, 5])
def test_equals_the_one_hot_route(cuda_device, C, B, F):
    # odd image sizes: partial warp tiles on both axes
    assert L.check_case(cuda_device, C, B, F, 157, 101, seed=C + 7 * B + F, close=0.5) > 0


@pytest.mark.parametrize("C", [14, 64])
@pytest.mark.parametrize("flags", [0, N.SPSG_FLAG_SMEM_MAPS])
def test_c3_size_28_warp_ctas(cuda_device, C, flags):
    """8 chunks x 5 views at 320x256: enough tiles for the 28-warp CTAs; maps through L1, and staged by TMA."""
    L.check_case(cuda_device, C, 8, 5, 320, 256, seed=C, flags=flags)


@pytest.mark.parametrize("flags", L.DEBUG_FLAGS)
@pytest.mark.parametrize("B", [1, 3])
def test_debug_flags(cuda_device, flags, B):
    L.check_case(cuda_device, 20, B, 2, 131, 97, seed=B + flags, flags=flags, close=0.5)


@pytest.mark.parametrize("kind", ["spheres", "soup"])
@pytest.mark.parametrize("B,F", [(1, 1), (2, 3)])
def test_grid_beyond_shared_memory_maps(cuda_device, kind, B, F):
    L.check_case(cuda_device, 41, B, F, 163, 125, seed=B * F, dims=L.BIG_DIMS, kind=kind)


@pytest.mark.parametrize("route", ["packed", "prebuilt"])
@pytest.mark.parametrize("B,F", [(1, 1), (3, 2)])
def test_index_routes(cuda_device, route, B, F):
    L.check_case(cuda_device, 14, B, F, 160, 128, seed=3 + B, route=route)
    L.check_case(cuda_device, 64, B, F, 99, 77, seed=5 + B, route=route, kind="soup")


def test_empty_chunks_and_views(cuda_device):
    L.check_case(cuda_device, 20, 3, 3, 160, 128, seed=11, empty=(1,), away=0.4)
    L.check_case(cuda_device, 20, 3, 1, 160, 128, seed=12, empty=(0, 2))
    L.check_case(cuda_device, 5, 1, 2, 64, 48, seed=13, away=1.0)


@pytest.mark.parametrize("C", [1, 14, 64])
def test_no_voxels(cuda_device, C):
    L.check_case(cuda_device, C, 2, 2, 80, 64, seed=C, n_zero=True)
    lab, hist = L.module(cuda_device, 1, 1, 80, 64, 0, C).render_labels(
        torch.zeros(0, 4, dtype=torch.int64, device=cuda_device), torch.zeros(0, 1, device=cuda_device),
        torch.zeros(0, dtype=torch.uint8, device=cuda_device), *L.cameras(cuda_device, 1, np.random.default_rng(0), 80, 64,
                                                                           S.DIMS_ZYX), histogram=True)
    assert bool((lab == C).all()) and hist.tolist() == [0] * C + [80 * 64]


@pytest.mark.parametrize("C", [1, 14, 41])
def test_labels_at_and_above_c(cuda_device, C):
    """Every voxel labelled C, or above C: every pixel is C, hit or not."""
    t, n, _ = L.D.room(cuda_device, 2, 4)
    view, intr = L.cameras(cuda_device, 2, np.random.default_rng(1), 96, 80, S.DIMS_ZYX)
    m = L.module(cuda_device, 2, 1, 96, 80, n, C)
    for v in (C, C + 1, 255):
        lab, hist = m.render_labels(t["locs"], t["sdf"], torch.full((n,), v, dtype=torch.uint8, device=cuda_device), view,
                                    intr, histogram=True)
        assert bool((lab == C).all()) and hist[C] == lab.numel() and int(hist[:C].sum()) == 0


def _payload(n, C, dev, seed):
    """(n, C) logits with the label maps' corner cases: NaN rows and entries, +inf, -inf in logit 0, -inf rows, exact ties
    (at, above and below 1), maxima of exactly 1 and of the float just below 1, all-zero rows."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    x = torch.randn(n, C, generator=g) * 2.0
    k = torch.randint(0, 12, (n,), generator=g)
    j = torch.randint(0, C, (n,), generator=g)
    below = float(np.nextafter(np.float32(1.0), np.float32(0.0)))
    x[k == 1, :] = float("nan")
    x[(k == 2), j[k == 2]] = float("nan")
    x[(k == 3), j[k == 3]] = float("inf")
    x[k == 4, 0] = -float("inf")
    x[k == 5, :] = -float("inf")
    x[k == 6, :] = 0.0
    s = k == 7
    x[s, :] = torch.clamp(x[s, :], max=0.5)
    x[s, j[s]] = 1.0
    s = k == 8
    x[s, :] = torch.clamp(x[s, :], max=0.5)
    x[s, j[s]] = below
    s = k == 9  # a tie of two maxima >= 1
    x[s, :] = torch.clamp(x[s, :], max=0.5)
    x[s, j[s]] = 3.0
    x[s, (j[s] + 1) % C] = 3.0
    s = k == 10  # a tie at exactly 1
    x[s, :] = torch.clamp(x[s, :], max=0.5)
    x[s, j[s]] = 1.0
    x[s, (j[s] + C // 2) % C] = 1.0
    return x.contiguous().to(dev)


@pytest.mark.parametrize("C", [1, 2, 14, 20, 41, 64])
@pytest.mark.parametrize("B,F", [(1, 1), (3, 3)])
def test_equals_the_logits_route(cuda_device, C, B, F):
    t, n, _ = L.D.room(cuda_device, B, C)
    view, intr = L.cameras(cuda_device, B * F, np.random.default_rng(C), 160, 128, S.DIMS_ZYX, close=0.5)
    logits = _payload(n, C, cuda_device, C + B)
    m = L.module(cuda_device, B, F, 160, 128, n, C)
    with torch.no_grad():
        _, _, _, sem = m(t["locs"], t["sdf"], t["color"], t["normal"], logits, view, intr)
        want = losses.labels_from_render(sem, histogram=True)
    got = m.render_labels(t["locs"], t["sdf"], losses.labels_from_render(logits), view, intr, histogram=True)
    L.compare(got, want, "logits route C=%d" % C)


def test_module_buffers_untouched_and_backward_raises(cuda_device):
    B, F, w, h, C = 2, 2, 120, 96, 20
    t, n, _ = L.D.room(cuda_device, B, 8)
    view, intr = L.cameras(cuda_device, B * F, np.random.default_rng(8), w, h, S.DIMS_ZYX, close=0.5)
    m = L.module(cuda_device, B, F, w, h, n, C)
    sem = torch.randn(n, C, device=cuda_device)
    leaves = [x.clone().requires_grad_(True) for x in (t["sdf"], t["color"], t["normal"], sem)]
    out = m(t["locs"], *leaves, view, intr)
    torch.cuda.synchronize()
    names = ("image_color", "image_depth", "image_normal", "image_semantic", "mapping3dto2d", "mapping3dto2d_num", "d_color",
             "d_depth", "d_normal", "d_semantic")
    before = {k: getattr(m, k).clone() for k in names}
    forwards = m.workspace.forwards
    lab = m.render_labels(t["locs"], t["sdf"], L.voxel_labels(n, C, 2, cuda_device), view, intr)
    torch.cuda.synchronize()
    assert lab.shape == (B * F, h, w) and lab.data_ptr() != m.image_semantic.data_ptr()
    for k in names:
        assert torch.equal(getattr(m, k).view(torch.uint8) if getattr(m, k).dtype == torch.float32 else getattr(m, k),
                           before[k].view(torch.uint8) if before[k].dtype == torch.float32 else before[k]), k
    assert m.workspace.forwards == forwards + 1
    # the autograd backward of the earlier render
    with pytest.raises(RuntimeError, match="backward after a later forward"):
        torch.autograd.grad(out, leaves, [torch.zeros_like(o) for o in out])
    # a raw backward on the module's workspace
    g = [torch.zeros_like(x) for x in (m.image_color, m.image_depth, m.image_normal, m.image_semantic)]
    with pytest.raises(RuntimeError, match="without a matching forward"):
        rc.backward(*g, m.sparse_mapping, m.mapping3dto2d, m.mapping3dto2d_num,
                    [B, S.DIMS_ZYX[2], S.DIMS_ZYX[1], S.DIMS_ZYX[0], n], m.d_color, m.d_depth, m.d_normal, m.d_semantic,
                    views_per_chunk=F, workspace_owner=m.workspace)
    # without a module: the workspace cached for sparse_mapping
    sm = torch.zeros_like(m.sparse_mapping)
    opts = [w, h, S.DEPTH_MIN, S.DEPTH_MAX, S.THRESH_SAMPLE_DIST, S.RAY_INCREMENT, S.DIMS_ZYX[2], S.DIMS_ZYX[1], S.DIMS_ZYX[0]]
    rc.forward(sm, t["locs"], t["sdf"], t["color"], t["normal"], leaves[3].detach(), view, m.image_color, m.image_depth,
               m.image_normal, m.image_semantic, m.mapping3dto2d, m.mapping3dto2d_num, intr, opts, views_per_chunk=F,
               build_index=True)
    raw = rc.render_labels(sm, t["locs"], t["sdf"], L.voxel_labels(n, C, 2, cuda_device), view, intr, opts, C,
                           views_per_chunk=F)
    assert torch.equal(raw, lab)
    with pytest.raises(RuntimeError, match="without a matching forward"):
        rc.backward(*g, sm, m.mapping3dto2d, m.mapping3dto2d_num, [B, S.DIMS_ZYX[2], S.DIMS_ZYX[1], S.DIMS_ZYX[0], n],
                    m.d_color, m.d_depth, m.d_normal, m.d_semantic, views_per_chunk=F)


@pytest.mark.parametrize("flags", [DET, ALL, DET | ALL, DET | N.SPSG_FLAG_GENERIC_SEMANTIC])
def test_module_flags_change_nothing(cuda_device, flags):
    B, F, w, h, C = 3, 2, 144, 112, 14
    t, n, _ = L.D.room(cuda_device, B, 2)
    view, intr = L.cameras(cuda_device, B * F, np.random.default_rng(2), w, h, S.DIMS_ZYX, close=0.5)
    labels = L.voxel_labels(n, C, 3, cuda_device)
    want = L.module(cuda_device, B, F, w, h, n, C).render_labels(t["locs"], t["sdf"], labels, view, intr, histogram=True)
    m = L.module(cuda_device, B, F, w, h, n, C, flags=flags & ~ALL, max_pixels=None if flags & ALL else 64)
    L.compare(m.render_labels(t["locs"], t["sdf"], labels, view, intr, histogram=True), want, "flags %#x" % flags)
    torch.use_deterministic_algorithms(True)
    try:
        L.compare(m.render_labels(t["locs"], t["sdf"], labels, view, intr, histogram=True), want, "torch deterministic")
    finally:
        torch.use_deterministic_algorithms(False)


def test_argument_checks(cuda_device):
    t, n, _ = L.D.room(cuda_device, 1, 0)
    view, intr = L.cameras(cuda_device, 1, np.random.default_rng(0), 80, 64, S.DIMS_ZYX)
    m = L.module(cuda_device, 1, 1, 80, 64, n, 14)
    lab = torch.zeros(n, dtype=torch.uint8, device=cuda_device)
    with pytest.raises(RuntimeError, match="voxel_labels must have dtype"):
        m.render_labels(t["locs"], t["sdf"], lab.long(), view, intr)
    with pytest.raises(RuntimeError, match="fewer than N"):
        m.render_labels(t["locs"], t["sdf"], lab[:-1], view, intr)
    with pytest.raises(RuntimeError, match="voxel_labels must be a CUDA tensor"):
        m.render_labels(t["locs"], t["sdf"], lab.cpu(), view, intr)
    with pytest.raises(RuntimeError, match="view_matrix has"):
        m.render_labels(t["locs"], t["sdf"], lab, torch.cat([view, view]), torch.cat([intr, intr]))


# ---- the training step's target labels (train.py:581-622)

def old_target_labels(self, target_for_sdf, target_for_colors, target_for_semantics, view_matrix, intrinsics, transform):
    """ViewGuidedTrainStep._target_labels before the label render: colours, normals and the one-hot semantics of the
    target rendered in full, labels from the C-wide image."""
    from spsg_b200 import normals, sparsify
    locs, vals = sparsify.sparsify_predictions(target_for_sdf, self.truncation)
    colors = target_for_colors[locs[:, 3], locs[:, 0], locs[:, 1], locs[:, 2], :].float() / 255.0
    if self.views == 1:
        target_normals = normals.compute_normals_sparse(locs, vals, self.dims3d, transform=transform)
    else:
        target_normals = normals.compute_normals_sparse(locs, vals, self.dims3d, num_chunks=self.batch_size)
    sem = sparsify.gather_dense(locs, target_for_semantics.float())
    onehot = Fn.one_hot(sem[:, 0].long(), self.num_classes + 1)[..., :-1].float().contiguous()
    _, _, _, raycast_semantic = self.raycaster(locs, vals, colors.contiguous(), target_normals, onehot, view_matrix,
                                               intrinsics)
    return losses.labels_from_render(raycast_semantic)


@pytest.mark.parametrize("C", [14, 41])
def test_target_labels_equal_the_old_route(cuda_device, C):
    from tests import fuzz_semantic_classes as Z
    torch.manual_seed(C)
    step = Z.train_step(cuda_device, Z.GenC(C).to(cuda_device), C, flags=0)
    s = Z.train_sample(cuda_device, C)
    tsdf, tcol = step.loss_util.compute_targets(s["sdf"], step.truncation, True, s.get("known"), s["colors"])
    args = (tsdf, tcol, s["semantics"], s["view_matrix"], s["images_intrinsic"], torch.inverse(s["view_matrix"]))
    with torch.no_grad():
        want = old_target_labels(step, *args).clone()
        got = step._target_labels(*args)
    assert got.shape == want.shape and torch.equal(got, want)
    assert int((got < C).sum()) > 0


_TRAIN_SCRIPT = r"""
import json, sys
import torch
sys.path.insert(0, %(root)r)
torch.backends.cudnn.benchmark = False
torch.use_deterministic_algorithms(True)
from spsg_b200 import train_step as T
from tests import fuzz_semantic_classes as Z
from tests import test_gpu_label_render as G
C = %(C)d
dev = torch.device("cuda", 0)
torch.manual_seed(1234)
base = Z.GenC(C).to(dev)
sample = Z.train_sample(dev, C)
new = T.ViewGuidedTrainStep._target_labels


class GradOnly:
    def __init__(self, model):
        self.model = model
    def zero_grad(self, set_to_none=True):
        self.model.zero_grad(set_to_none=True)
    def step(self):
        pass

out = []
for route in (new, G.old_target_labels):
    T.ViewGuidedTrainStep._target_labels = route
    model = Z.GenC(C).to(dev)
    model.load_state_dict(base.state_dict())
    step = Z.train_step(dev, model, C, flags=0)
    loss = step({k: (v.clone() if v is not None else None) for k, v in sample.items()}, optimizer=GradOnly(model))
    torch.cuda.synchronize()
    out.append(dict(loss=float(loss), n=step.last["num_locs"],
                    bits=torch.cat([p.grad.reshape(-1) for p in model.parameters()]).view(torch.int32).tolist()))
T.ViewGuidedTrainStep._target_labels = new
a, b = out
print(json.dumps(dict(loss=[a["loss"], b["loss"]], same_loss=a["loss"] == b["loss"], n=a["n"],
                      differing_grads=sum(x != y for x, y in zip(a["bits"], b["bits"])), grads=len(a["bits"]))))
"""


@pytest.mark.parametrize("C", [14, 41])
def test_train_step_equals_the_old_route_bit_for_bit(cuda_device, C):
    """Under torch.use_deterministic_algorithms(True), with a seeded stand-in generator, the step's loss and every parameter
    gradient are bit-identical to the same step with the previous _target_labels patched in."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, CUBLAS_WORKSPACE_CONFIG=":4096:8")
    out = subprocess.run([sys.executable, "-c", _TRAIN_SCRIPT % dict(root=root, C=C)], cwd=root, env=env,
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-4000:]
    r = json.loads(out.stdout.strip().splitlines()[-1])
    print("C=%d train step, label render vs one-hot render:" % C, r)
    assert r["n"] > 0 and r["same_loss"] and r["differing_grads"] == 0, r


# ---- the room driver

def old_render_room(predict, room_dims_zyx, device, views_per_chunk=5, chunks_per_launch=8, chunk_yx=(64, 64), stride=32,
                    width=S.WIDTH, height=S.HEIGHT, rank=0, world=1, max_num_locs_per_sample=640000, keep_images=True):
    """room.render_room before the label render: normals, the full render, labels_from_render of the semantic image."""
    from spsg_b200 import parallel as P
    from spsg_b200 import room as R
    from spsg_b200.normals import compute_normals_sparse
    from spsg_b200.raycast_rgbd import RaycastRGBD
    dz = room_dims_zyx[0]
    chunk_dims = (dz, chunk_yx[0], chunk_yx[1])
    windows = R.chunk_windows(room_dims_zyx, chunk_yx, stride)
    mine = [windows[i] for i in P.shard_round_robin(len(windows), rank, world)]
    B, F = chunks_per_launch, views_per_chunk
    rcm = RaycastRGBD(B, chunk_dims, width, height, S.DEPTH_MIN, S.DEPTH_MAX, S.THRESH_SAMPLE_DIST, S.RAY_INCREMENT,
                      max_num_frames=F, max_num_locs_per_sample=max_num_locs_per_sample, device=device)
    view_np, intr_np = R.window_views(F, chunk_dims)
    view = torch.from_numpy(np.tile(view_np, (B, 1, 1))).to(device)
    intr = torch.from_numpy(np.tile(intr_np, (B, 1))).to(device)
    grid2cam = torch.inverse(view[::F]).contiguous()
    hist = torch.zeros(S.NUM_CLASSES + 1, dtype=torch.int64, device=device)
    images = []
    predict_group = getattr(predict, "predict_group", None)
    for s in range(0, len(mine), B):
        group = mine[s:s + B]
        if predict_group is not None:
            locs, sdf, color, sem = predict_group(group, chunk_yx)
            edges = torch.searchsorted(locs[:, 3].contiguous(), torch.arange(len(group) + 1, device=device)).tolist()
            present = [b for b in range(len(group)) if edges[b + 1] > edges[b]]
            slots = len(group)
        else:
            parts = [predict(y0, x0, chunk_yx) for (y0, x0) in group]
            present = [k for k, p in enumerate(parts) if p[0].shape[0] > 0]
            slots = len(present)
            if present:
                locs = torch.cat([torch.cat([parts[k][0], torch.full((parts[k][0].shape[0], 1), b, dtype=torch.long,
                                                                     device=device)], 1)
                                  for b, k in enumerate(present)]).contiguous()
                sdf = torch.cat([parts[k][1] for k in present])
                color = torch.cat([parts[k][2] for k in present])
                sem = torch.cat([parts[k][3] for k in present])
        if not present:
            continue
        with torch.no_grad():
            normals = compute_normals_sparse(locs, sdf, chunk_dims, grid2cam, num_chunks=B)
            _, _, _, sem_img = rcm(locs, sdf, color, normals, sem, view, intr)
            labels, h = losses.labels_from_render(sem_img[:slots * F], histogram=True)
            labels = labels.view(slots, F, height, width)
            if len(present) < slots:
                h[S.NUM_CLASSES] -= (slots - len(present)) * F * width * height
                labels = labels[torch.tensor(present, device=device)]
            hist += h
        if keep_images:
            for j, k in enumerate(present):
                images.append((group[k], labels[j].cpu()))
    return hist.cpu().numpy().astype(np.float64), images


@pytest.mark.parametrize("grouped", [True, False])
def test_room_driver_equals_the_old_route(cuda_device, grouped):
    """Labels and histogram of render_room against the previous route: a room with empty windows (idle slots in a launch
    group), a last group shorter than the launch, one rank and two ranks."""
    from spsg_b200 import room as R
    dims = (64, 96, 160)
    room = R.synthetic_room_sdf(dims, cuda_device, seed=7)
    room[:, :, 96:] = 2.0 * S.TRUNCATION + 1.0  # the windows over x >= 96 hold no voxel
    predict = R.synthetic_predictor(room)
    if not grouped:
        group_predict = predict
        predict = lambda y0, x0, chunk_yx: group_predict(y0, x0, chunk_yx)  # noqa: E731  (no predict_group: packed slots)
    kw = dict(views_per_chunk=3, width=96, height=72, max_num_locs_per_sample=200000)
    for world, cpl in ((1, 4), (2, 3)):
        for rank in range(world):
            got = R.render_room(predict, dims, cuda_device, chunks_per_launch=cpl, rank=rank, world=world, keep_images=True,
                                **kw)
            want_hist, want_images = old_render_room(predict, dims, cuda_device, chunks_per_launch=cpl, rank=rank,
                                                     world=world, **kw)
            np.testing.assert_array_equal(got["label_hist"], want_hist)
            assert [w for w, _ in got["images"]] == [w for w, _ in want_images]
            for (w, a), (_, b) in zip(got["images"], want_images):
                assert torch.equal(a, b), "window %s" % (w,)
            assert got["label_hist"].sum() == got["rays"] and got["label_hist"][:S.NUM_CLASSES].sum() > 0


def test_fuzz_slice(cuda_device):
    failures = L.sweep(cuda_device, cases=16, seed=2026)
    assert not failures, failures
