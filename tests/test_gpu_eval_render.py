"""Eval render (``losses.evaluate_2d``, spsg_raycast_eval):
  * loss terms against the fused forward (normalisers bit for bit, terms within 1e-6) and the literal PyTorch expressions,
    label map and confusion matrix against labels_from_render of the forward's semantic image, on every route: C 1-64,
    B 1-8, F 1-5, terms switched off, weights, labels at and above C, N = 0, empty chunks and views, int64 / packed /
    prebuilt rows, 28-warp CTAs with both map paths, a grid beyond shared-memory maps, the generic kernels at C = 14;
  * label corner cases of the logits (NaN, +-inf, ties, maxima at and just below 1);
  * determinism across calls, debug flags, modes and all-pixels modules; module isolation; argument checks;
  * ``semantic_metrics`` against numpy, and ``ViewGuidedTrainStep.validate`` against ``__call__``.
Helpers and the random sweep: tests/fuzz_eval_render.py."""
import numpy as np
import pytest
import torch

from spsg_b200 import _native as N
from spsg_b200 import losses
from spsg_b200 import raycast_rgbd_cuda as rc
from spsg_b200 import synthetic as S
from tests import fuzz_eval_render as E
from tests import fuzz_label_render as L

pytestmark = pytest.mark.gpu

DET, ALL = N.SPSG_FLAG_DETERMINISTIC, N.SPSG_FLAG_ALL_PIXELS


@pytest.mark.parametrize("C", [1, 2, 14, 20, 41, 64])
@pytest.mark.parametrize("B", [1, 3, 8])
@pytest.mark.parametrize("F", [1, 3, 5])
def test_equals_the_fused_forward(cuda_device, C, B, F):
    assert E.check_case(cuda_device, C, B, F, 157, 101, seed=C + 7 * B + F, close=0.5) > 0


@pytest.mark.parametrize("terms", [(), ("depth",), ("color",), ("semantic",), ("depth", "color"), ("color", "semantic")])
@pytest.mark.parametrize("weights", [(True, True), (False, False)])
def test_terms_and_weights(cuda_device, terms, weights):
    E.check_case(cuda_device, 20, 2, 2, 120, 96, seed=len(terms), terms=terms, weight_color=weights[0],
                 class_weight=weights[1], close=0.5)


@pytest.mark.parametrize("C", [14, 64])
@pytest.mark.parametrize("flags", [0, N.SPSG_FLAG_SMEM_MAPS])
def test_c3_size_28_warp_ctas(cuda_device, C, flags):
    E.check_case(cuda_device, C, 8, 5, 320, 256, seed=C, flags=flags)


@pytest.mark.parametrize("flags", L.DEBUG_FLAGS)
def test_debug_flags(cuda_device, flags):
    E.check_case(cuda_device, 20, 3, 2, 131, 97, seed=3 + flags, flags=flags, close=0.5)


@pytest.mark.parametrize("kind", ["spheres", "soup"])
def test_grid_beyond_shared_memory_maps(cuda_device, kind):
    E.check_case(cuda_device, 41, 2, 2, 163, 125, seed=5, dims=E.BIG_DIMS, kind=kind)


@pytest.mark.parametrize("route", ["packed", "prebuilt"])
@pytest.mark.parametrize("C", [14, 64])
def test_index_routes(cuda_device, route, C):
    E.check_case(cuda_device, C, 3, 2, 160, 128, seed=3 + C, route=route)


def test_empty_chunks_views_and_no_voxels(cuda_device):
    E.check_case(cuda_device, 20, 3, 3, 160, 128, seed=11, empty=(1,), away=0.4)
    E.check_case(cuda_device, 5, 1, 2, 64, 48, seed=13, away=1.0)
    for C in (1, 14, 64):
        E.check_case(cuda_device, C, 2, 2, 80, 64, seed=C, n_zero=True)


def test_generic_kernels_at_14(cuda_device):
    """The fused forward's C-generic epilogue at C = 14 (SPSG_FLAG_GENERIC_SEMANTIC) against the eval epilogue."""
    E.check_case(cuda_device, 14, 3, 2, 160, 128, seed=21, generic=True)


def _literal(imgs, tg, C, voxelsize=0.02, weights=(1.0, 0.7, 0.3)):
    """train.py:635-638, loss.py:246-257, train.py:744-746 on the renderings, in float64."""
    color, depth, sem = (x.double() for x in imgs)
    td, tc, wc, tl, cw = tg
    hit = depth != -float("inf")
    out = []
    m = hit & (td != 0)
    out.append((depth[m] * voxelsize - td.double()[m]).abs().mean())
    w = wc.double()[..., None] if wc is not None else torch.ones_like(depth)[..., None]
    out.append((color * w - tc.double() * w).abs()[hit].mean())
    valid = hit & (tl.long() < C) & (sem[..., 0] != -float("inf"))
    y = tl.long()[valid]
    nll = -torch.log_softmax(sem[valid], -1).gather(1, y[:, None])[:, 0]
    cwt = cw.double()[y] if cw is not None else torch.ones_like(nll)
    out.append((cwt * nll).sum() / cwt.sum())
    return torch.stack(out)


@pytest.mark.parametrize("C", [1, 14, 41])
def test_terms_equal_the_literal_expressions(cuda_device, C):
    B, F, w, h = 2, 2, 120, 96
    t, n, _ = L.D.room(cuda_device, B, C)
    view, intr = L.cameras(cuda_device, B * F, np.random.default_rng(C), w, h, S.DIMS_ZYX, close=0.5)
    color, logits = E.payload(n, C, C, cuda_device)
    tg = E.targets(B * F, h, w, C, C + 1, cuda_device)
    _, _, _, imgs = E.reference(L.module(cuda_device, B, F, w, h, n, C), t["locs"], t["sdf"], color, logits, view, intr, tg)
    total, terms, _, _ = E.evaluate(L.module(cuda_device, B, F, w, h, n, C), t["locs"], t["sdf"], color, logits, view,
                                    intr, tg)
    lit = _literal(imgs, tg, C)
    assert torch.allclose(terms.double(), lit, rtol=1e-5, atol=0), (terms.tolist(), lit.tolist())
    assert abs(float(total) - float((lit * torch.tensor([1.0, 0.7, 0.3], dtype=torch.float64, device=lit.device)).sum())) \
        <= 1e-5 * abs(float(total))


def _payload(n, C, dev, seed):
    from tests.test_gpu_label_render import _payload as corner_cases
    return corner_cases(n, C, dev, seed)


@pytest.mark.parametrize("C", [1, 2, 14, 41, 64])
def test_labels_of_corner_case_logits(cuda_device, C):
    """NaN rows and entries, +-inf, -inf in logit 0, exact ties, maxima of 1 and just below 1: the label map and the
    confusion matrix equal labels_from_render of the forward's image; the losses match too (NaN where the forward's is)."""
    B, F, w, h = 3, 3, 160, 128
    t, n, _ = L.D.room(cuda_device, B, C)
    view, intr = L.cameras(cuda_device, B * F, np.random.default_rng(C), w, h, S.DIMS_ZYX, close=0.5)
    logits = _payload(n, C, cuda_device, C + B)
    color, _ = E.payload(n, C, C, cuda_device)
    tg = E.targets(B * F, h, w, C, C + 2, cuda_device)
    want = E.reference(L.module(cuda_device, B, F, w, h, n, C), t["locs"], t["sdf"], color, logits, view, intr, tg)
    got = E.evaluate(L.module(cuda_device, B, F, w, h, n, C), t["locs"], t["sdf"], color, logits, view, intr, tg)
    E.compare(got, want, "corner cases C=%d" % C)
    assert int((got[3] < C).sum()) > 0


def test_deterministic_across_calls_flags_and_modes(cuda_device):
    B, F, w, h, C = 3, 2, 144, 112, 20
    t, n, _ = L.D.room(cuda_device, B, 2)
    view, intr = L.cameras(cuda_device, B * F, np.random.default_rng(2), w, h, S.DIMS_ZYX, close=0.5)
    color, logits = E.payload(n, C, 4, cuda_device)
    tg = E.targets(B * F, h, w, C, 5, cuda_device)

    def run(m):
        total, terms, conf, lab = E.evaluate(m, t["locs"], t["sdf"], color, logits, view, intr, tg)
        return E.loss_block(total, terms).clone(), conf.clone(), lab.clone()
    base = run(L.module(cuda_device, B, F, w, h, n, C))
    results = []
    m = L.module(cuda_device, B, F, w, h, n, C)
    results += [run(m) for _ in range(3)]
    for flags in L.DEBUG_FLAGS + (DET, DET | N.SPSG_FLAG_GENERIC_SEMANTIC):
        results.append(run(L.module(cuda_device, B, F, w, h, n, C, flags=flags)))
    results.append(run(L.module(cuda_device, B, F, w, h, n, C, max_pixels=None)))
    torch.use_deterministic_algorithms(True)
    try:
        results.append(run(m))
    finally:
        torch.use_deterministic_algorithms(False)
    for k, r in enumerate(results):
        assert torch.equal(r[0].view(torch.int32), base[0].view(torch.int32)), (k, r[0].tolist(), base[0].tolist())
        assert torch.equal(r[1], base[1]) and torch.equal(r[2], base[2]), k


def test_module_buffers_untouched_and_backward_raises(cuda_device):
    B, F, w, h, C = 2, 2, 120, 96, 20
    t, n, _ = L.D.room(cuda_device, B, 8)
    view, intr = L.cameras(cuda_device, B * F, np.random.default_rng(8), w, h, S.DIMS_ZYX, close=0.5)
    m = L.module(cuda_device, B, F, w, h, n, C)
    color, logits = E.payload(n, C, 9, cuda_device)
    leaves = [x.clone().requires_grad_(True) for x in (t["sdf"], color, t["normal"], logits)]
    out = m(t["locs"], *leaves, view, intr)
    torch.cuda.synchronize()
    names = ("image_color", "image_depth", "image_normal", "image_semantic", "mapping3dto2d", "mapping3dto2d_num", "d_color",
             "d_depth", "d_normal", "d_semantic")
    before = {k: getattr(m, k).clone() for k in names}
    forwards = m.workspace.forwards
    tg = E.targets(B * F, h, w, C, 10, cuda_device)
    total, terms, conf, lab = E.evaluate(m, t["locs"], t["sdf"], color, logits, view, intr, tg)
    assert not total.requires_grad and not terms.requires_grad
    for k in names:
        a, b = getattr(m, k), before[k]
        assert torch.equal(a.view(torch.uint8) if a.dtype == torch.float32 else a,
                           b.view(torch.uint8) if b.dtype == torch.float32 else b), k
    assert m.workspace.forwards == forwards + 1
    with pytest.raises(RuntimeError, match="backward after a later forward"):
        torch.autograd.grad(out, leaves, [torch.zeros_like(o) for o in out])
    g = [torch.zeros_like(x) for x in (m.image_color, m.image_depth, m.image_normal, m.image_semantic)]
    with pytest.raises(RuntimeError, match="without a matching forward"):
        rc.backward(*g, m.sparse_mapping, m.mapping3dto2d, m.mapping3dto2d_num,
                    [B, S.DIMS_ZYX[2], S.DIMS_ZYX[1], S.DIMS_ZYX[0], n], m.d_color, m.d_depth, m.d_normal, m.d_semantic,
                    views_per_chunk=F, workspace_owner=m.workspace)
    # without target labels: no confusion matrix; without labels=True: no label map
    _, _, conf2, lab2 = losses.evaluate_2d(m, t["locs"], t["sdf"], color, logits, view, intr, images_depth=tg[0])
    assert conf2 is None and lab2 is None


def test_argument_checks(cuda_device):
    t, n, _ = L.D.room(cuda_device, 1, 0)
    view, intr = L.cameras(cuda_device, 1, np.random.default_rng(0), 80, 64, S.DIMS_ZYX)
    m = L.module(cuda_device, 1, 1, 80, 64, n, 14)
    color, logits = E.payload(n, 14, 0, cuda_device)
    with pytest.raises(RuntimeError, match="vals_semantics must be"):
        losses.evaluate_2d(m, t["locs"], t["sdf"], color, logits[:, :13].contiguous(), view, intr)
    with pytest.raises(RuntimeError, match="vals_colors must have dtype"):
        losses.evaluate_2d(m, t["locs"], t["sdf"], color.double(), logits, view, intr)
    with pytest.raises(RuntimeError, match="view_matrix has"):
        losses.evaluate_2d(m, t["locs"], t["sdf"], color, logits, torch.cat([view, view]), torch.cat([intr, intr]))
    with pytest.raises(RuntimeError, match="target_label must be"):
        losses.evaluate_2d(m, t["locs"], t["sdf"], color, logits, view, intr,
                           target2d_label=torch.zeros(1, 64, 80, dtype=torch.int64, device=cuda_device))


@pytest.mark.parametrize("C", [1, 5, 20])
def test_semantic_metrics_equal_numpy(cuda_device, C):
    rng = np.random.default_rng(C)
    conf = rng.integers(0, 50, (C + 1, C + 1))
    if C > 2:
        conf[1, :] = 0
        conf[:, 1] = 0  # a class with an empty union
    acc, iou, miou = losses.semantic_metrics(torch.from_numpy(conf).to(cuda_device))
    m = conf[:C].astype(np.float64)
    tp = np.diag(m[:, :C])
    union = m.sum(1) + m[:, :C].sum(0) - tp
    with np.errstate(invalid="ignore", divide="ignore"):
        want_iou = tp / union
    assert abs(float(acc) - tp.sum() / m.sum()) < 1e-12
    np.testing.assert_allclose(iou.cpu().numpy(), want_iou, rtol=1e-12, equal_nan=True)
    assert abs(float(miou) - want_iou[union > 0].mean()) < 1e-12


_VALIDATE_SCRIPT = r"""
import json, sys
import torch
sys.path.insert(0, %(root)r)
torch.backends.cudnn.benchmark = False
torch.use_deterministic_algorithms(True)
from spsg_b200 import losses
from spsg_b200 import train_step as T
from tests import fuzz_semantic_classes as Z
C = %(C)d
dev = torch.device("cuda", 0)
torch.manual_seed(1234)
base = Z.GenC(C).to(dev)
sample = Z.train_sample(dev, C)
clone = lambda: {k: (v.clone() if v is not None else None) for k, v in sample.items()}
model = Z.GenC(C).to(dev)
model.load_state_dict(base.state_dict())
step = Z.train_step(dev, model, C, flags=0)
step(clone())
torch.cuda.synchronize()
ref = dict(step.last)
model.zero_grad(set_to_none=True)
val_total = step.validate(clone())
torch.cuda.synchronize()
got = dict(step.last)
grads = sum(p.grad is not None for p in model.parameters())
# the literal confusion: target labels of the label render, labels_from_render of the prediction's render
s = clone()
lu, Tr = step.loss_util, step.truncation
with torch.no_grad():
    tsdf, tcol = lu.compute_targets(s["sdf"], Tr, True, s.get("known"), s["colors"])
    occ, sdf, col, sem = model(s["input"], s["mask"], pred_sdf=[True, True], pred_color=True, pred_semantic=True)
    empty = torch.sigmoid(occ) < 0.5
    tl = step._target_labels(tsdf, tcol, s["semantics"], s["view_matrix"], s["images_intrinsic"], None).clone()
    from spsg_b200 import sparsify
    locs, sv, cv, mv = sparsify.sparsify_predictions(sdf, Tr, empty, col, sem)
    normals = torch.zeros(locs.shape[0], 3, device=dev)
    _, _, _, img = step.raycaster(locs, sv, (cv + 1) * 0.5, normals, mv, s["view_matrix"], s["images_intrinsic"])
    lab = losses.labels_from_render(img)
    want = torch.bincount(tl.long().clamp(max=C).flatten() * (C + 1) + lab.long().flatten(), minlength=(C + 1) ** 2)
rel = lambda a, b: float(((a.double() - b.double()).abs() / b.double().abs().clamp(min=1e-30)).max())
print(json.dumps(dict(n=[ref["num_locs"], got["num_locs"]], occ=float(ref["loss_occ"]) == float(got["loss_occ"]),
                      sdf=float(ref["loss_sdf"]) == float(got["loss_sdf"]), terms_rel=rel(got["terms2d"], ref["terms2d"]),
                      confusion=bool(torch.equal(got["confusion"].flatten(), want)), grads=grads,
                      labelled=int((tl < C).sum()), total=float(val_total))))
"""


@pytest.mark.parametrize("C", [14, 41])
def test_validate_equals_the_training_step(cuda_device, C):
    """Under torch.use_deterministic_algorithms(True), with a seeded stand-in generator: validate's 3D losses and voxel count
    equal __call__'s, its 2D terms are within 1e-6, its confusion matrix is the literal one, and no .grad appears."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, CUBLAS_WORKSPACE_CONFIG=":4096:8")
    out = subprocess.run([sys.executable, "-c", _VALIDATE_SCRIPT % dict(root=root, C=C)], cwd=root, env=env,
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-4000:]
    r = json.loads(out.stdout.strip().splitlines()[-1])
    print("C=%d validate vs train step:" % C, r)
    assert r["n"][0] == r["n"][1] > 0 and r["occ"] and r["sdf"], r
    assert r["terms_rel"] <= 1e-6 and r["confusion"] and r["grads"] == 0 and r["labelled"] > 0, r


def test_fuzz_slice(cuda_device):
    failures = E.sweep(cuda_device, cases=16, seed=2027)
    assert not failures, failures
