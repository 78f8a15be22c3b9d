"""The producer glue on the heads a generator in channels_last_3d and/or under bfloat16 autocast produces: float32 and
bfloat16 heads, NCDHW, NDHWC and channel slices, read in place.  Rows, values and gradients against the literal
expressions of train.py:494-509 (with ``.float()`` on the gathered values), bit for bit; the indexed route; the
training step with ``autocast_bf16``."""
import types

import pytest
import torch
import torch.nn.functional as Fn

from tests.fuzz_head_formats import bits, fuzz_run, literal_gather, literal_locs, same_bits, same_values

pytestmark = pytest.mark.gpu


def _volume(shape, device, seed, channels=1, scale=3.0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(shape[0], channels, *shape[1:], generator=g) * scale).to(device)


def _layout(t, layout):
    if layout == "ncdhw":
        return t.contiguous()
    if layout == "ndhwc":
        return t.contiguous(memory_format=torch.channels_last_3d)
    # layout == "slice19": channels [lo, lo + C) of a 19-channel NDHWC tensor
    B, C = t.shape[:2]
    lo = 19 - C if C < 19 else 0
    wide = torch.full((B, 19) + tuple(t.shape[2:]), 7.0, dtype=t.dtype, device=t.device)
    wide = wide.contiguous(memory_format=torch.channels_last_3d)
    wide[:, lo:lo + C] = t
    return wide[:, lo:lo + C]


# ---- compaction -------------------------------------------------------------------------------------------------------

def _special_sdf(shape, device, seed, truncation):
    """random bfloat16 SDF with NaN, +-inf, +-0 and values at the (bf16-rounded) truncation and one ulp either side"""
    sdf = _volume(shape, device, seed)
    flat = sdf.view(-1)
    tb = float(torch.tensor(truncation).to(torch.bfloat16).float())
    ulp = 2.0 ** (torch.floor(torch.log2(torch.tensor(tb))).item() - 7)
    for k, v in enumerate([float("nan"), float("inf"), -float("inf"), 0.0, -0.0, tb, -tb, tb - ulp, -(tb - ulp),
                           tb + ulp, -(tb + ulp), truncation, -truncation]):
        flat[k::53] = v
    return sdf.to(torch.bfloat16)


@pytest.mark.parametrize("shape", [(1, 5, 7, 9), (2, 33, 31, 65), (3, 16, 16, 16), (5, 7, 13, 11), (8, 64, 32, 32)])
@pytest.mark.parametrize("use_empty", [False, True])
@pytest.mark.parametrize("layout", ["ncdhw", "ndhwc"])
def test_bf16_rows_match_nonzero(cuda_device, shape, use_empty, layout):
    from spsg_b200 import sparsify
    for T in (3.0, 3.005, 0.7):       # 3.005 and 0.7 are not bfloat16 values
        sdf = _layout(_special_sdf(shape, cuda_device, 1, T), layout)
        empty = (_volume(shape, cuda_device, 2) > 1.0) if use_empty else None
        got = sparsify.sparse_locs(sdf, T, empty)
        want = literal_locs(sdf, T, empty)
        assert got.dtype == torch.int64 and got.shape == want.shape and got.shape[0] > 0
        assert torch.equal(got, want), T
        counted = sparsify.count_locs(sdf, T, empty)
        assert counted.n == want.shape[0]
        assert torch.equal(sparsify.sparse_locs(sdf, T, empty, counted=counted), want)


def test_bf16_truncation_is_rounded_like_torch(cuda_device):
    """torch compares bf16 |sdf| with a Python scalar in bf16: 3.005 becomes 3.0, so a cell holding 3.0 is excluded
    although 3.0 < 3.005 -- the compaction does the same."""
    from spsg_b200 import sparsify
    sdf = torch.zeros(1, 1, 4, 4, 4, device=cuda_device, dtype=torch.bfloat16) + 10
    sdf[0, 0, 1, 2, 3] = 3.0
    sdf[0, 0, 2, 2, 2] = -2.984375                         # the bf16 value just below 3.0
    assert literal_locs(sdf, 3.005).tolist() == [[2, 2, 2, 0]]
    assert sparsify.sparse_locs(sdf, 3.005).tolist() == [[2, 2, 2, 0]]
    assert sparsify.sparse_locs(sdf.float(), 3.005).tolist() == [[1, 2, 3, 0], [2, 2, 2, 0]]   # float32: not rounded


def test_bf16_counted_checks(cuda_device):
    from spsg_b200 import sparsify
    sdf = _volume((2, 24, 16, 20), cuda_device, 11).to(torch.bfloat16)
    counted = sparsify.count_locs(sdf, 2.5)
    with pytest.raises(RuntimeError):
        sparsify.sparse_locs(sdf, 2.0, counted=counted)
    with pytest.raises(RuntimeError):
        sparsify.sparse_locs(sdf.clone(), 2.5, counted=counted)
    with pytest.raises(RuntimeError):
        sparsify.sparse_locs(sdf.float(), 2.5, counted=counted)
    sdf[0, 0, 0, 0, 0] = 0.0
    with pytest.raises(RuntimeError):
        sparsify.sparse_locs(sdf, 2.5, counted=counted)


# ---- gather and scatter -----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("layout", ["ncdhw", "ndhwc", "slice19"])
def test_gather_and_scatter_bit_identical(cuda_device, dtype, layout):
    from spsg_b200 import sparsify
    shape = (3, 13, 17, 19)
    locs = literal_locs(_volume(shape, cuda_device, 4), 2.5)
    heads = []
    for k, C in enumerate((1, 3, 14, 19)):
        v = _volume(shape, cuda_device, 10 + k, channels=C)
        v.view(-1)[::41] = float("nan")
        heads.append(_layout(v.to(dtype), layout))
    mine = [h.detach().requires_grad_(True) for h in heads]
    ref = [h.detach().clone().requires_grad_(True) for h in heads]
    got = sparsify.gather_dense(locs, *mine)
    want = [literal_gather(h, locs) for h in ref]
    for a, b in zip(got, want):
        assert a.dtype == torch.float32 and a.shape == b.shape
        assert torch.equal(bits(a), bits(b))
    g = torch.Generator(device="cpu").manual_seed(9)
    ws = [torch.randn(b.shape, generator=g).to(cuda_device) for b in want]
    for w in ws:
        w.view(-1)[::7] = -0.0
        w.view(-1)[1::97] = float("nan")
    # autograd.grad: the gradients as the backward returns them (a leaf's .grad would be re-laid out)
    ga = torch.autograd.grad(sum((a * w).sum() for a, w in zip(got, ws)), mine)
    gb = torch.autograd.grad(sum((b * w).sum() for b, w in zip(want, ws)), ref)
    for h, a, b in zip(heads, ga, gb):
        assert a.dtype == dtype
        if layout != "ncdhw" and h.shape[1] > 1:
            assert a.is_contiguous(memory_format=torch.channels_last_3d)
        if dtype == torch.float32 and h.is_contiguous():   # the original scatter (it keeps -0 as -0); NCDHW, or
            assert same_values(a, b)                      # NDHWC with one channel, which is the same memory order
        else:
            assert same_bits(a, b)


def test_more_than_four_mixed_heads(cuda_device):
    from spsg_b200 import sparsify
    shape = (2, 9, 10, 11)
    locs = literal_locs(_volume(shape, cuda_device, 5), 2.0)
    heads = [_layout(_volume(shape, cuda_device, 20 + k, channels=C).to(dt), lay)
             for k, (C, dt, lay) in enumerate([(3, torch.bfloat16, "ndhwc"), (14, torch.float32, "ncdhw"),
                                               (1, torch.bfloat16, "ncdhw"), (5, torch.float32, "slice19"),
                                               (19, torch.bfloat16, "slice19"), (2, torch.float32, "ndhwc"),
                                               (7, torch.bfloat16, "slice19")])]
    mine = [h.detach().requires_grad_(True) for h in heads]
    ref = [h.detach().clone().requires_grad_(True) for h in heads]
    got = sparsify.gather_dense(locs, *mine)
    want = [literal_gather(h, locs) for h in ref]
    for a, b in zip(got, want):
        assert torch.equal(bits(a), bits(b))
    sum((a * (k + 1.5)).sum() for k, a in enumerate(got)).backward()
    sum((b * (k + 1.5)).sum() for k, b in enumerate(want)).backward()
    for a, b in zip(mine, ref):
        assert a.grad.dtype == a.dtype and torch.equal(a.grad, b.grad)


def test_other_dtypes_are_rejected(cuda_device):
    from spsg_b200 import sparsify
    shape = (1, 4, 4, 4)
    sdf = _volume(shape, cuda_device, 1)
    locs = literal_locs(sdf, 2.0)
    for dt in (torch.float16, torch.int32, torch.float64):
        with pytest.raises(RuntimeError, match=str(dt)):
            sparsify.sparse_locs(sdf.to(dt), 2.0)
        with pytest.raises(RuntimeError, match=str(dt)):
            sparsify.gather_dense(locs, _volume(shape, cuda_device, 2, channels=3).to(dt))


# ---- the indexed route ------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("fused", [False, True])
def test_bf16_direct_feed_equals_the_locs_round_trip(cuda_device, fused):
    """sparsify_predictions(..., raycaster=m) on bf16 NDHWC heads: the compaction writes m's index and the widened SDF
    brick; renderings, index and counters must equal the plain int64 route over the same rows and values."""
    from spsg_b200 import losses, normals, sparsify, synthetic as S
    from tests.common import views
    from tests.test_gpu_sparsify import _dense_heads, _raycaster
    B, F = 2, 2
    sdf, col, sem = (_layout(t.to(torch.bfloat16), "ndhwc") for t in _dense_heads(cuda_device, [0, 1]))
    sem = _layout(sem, "slice19")
    _, _, view, intr = views(B, F, cuda_device, seed=3)
    g = torch.Generator(device="cpu").manual_seed(1)
    t_depth = (torch.rand(B * F, S.HEIGHT, S.WIDTH, generator=g) * 3.0).to(cuda_device)
    t_color = torch.rand(B * F, S.HEIGHT, S.WIDTH, 3, generator=g).to(cuda_device)
    t_label = torch.randint(0, 15, (B * F, S.HEIGHT, S.WIDTH), generator=g).to(torch.uint8).to(cuda_device)
    out = []
    for feed in (True, False):
        m = _raycaster(B, F, cuda_device, 200000)
        heads = [t.detach().requires_grad_(True) for t in (sdf, col, sem)]
        locs, v_sdf, v_col, v_sem = sparsify.sparsify_predictions(heads[0], S.TRUNCATION, None, heads[1], heads[2],
                                                                  raycaster=m if feed else None)
        assert (m.workspace._prebuilt is not None) == feed
        nrm = normals.compute_normals_sparse(locs, v_sdf.detach(), S.DIMS_ZYX, transform=torch.inverse(view[::F]),
                                             num_chunks=B)
        if fused:
            total, _, _ = losses.render_with_2d_losses(m, locs, v_sdf, v_col, nrm, v_sem, view, intr, images_depth=t_depth,
                                                       images_color=t_color, target2d_label=t_label, voxelsize=S.VOXELSIZE)
        else:
            c, d, nn, s = m(locs, v_sdf, v_col, nrm, v_sem, view, intr)
            hit = d != -float("inf")
            total = d[hit].sum() * 0.01 + c[hit].sum() + s[hit].sum() * 0.1
        total.backward()
        out.append((locs, m.sparse_mapping.clone(), m.image_color.clone(), m.image_depth.clone(), m.image_normal.clone(),
                    m.image_semantic.clone(), m.mapping3dto2d_num[:locs.shape[0] * F].clone(), total.detach().clone(),
                    heads[0].grad.float(), heads[1].grad.float(), heads[2].grad.float()))
        assert heads[1].grad.dtype == torch.bfloat16
        assert heads[1].grad.is_contiguous(memory_format=torch.channels_last_3d)
    names = ("locs", "sparse_mapping", "color", "depth", "normal", "semantic", "mapping3dto2d_num", "loss", "d_sdf", "d_color",
             "d_semantic")
    for a, b, name in zip(out[0], out[1], names):
        if name.startswith("d_") or name == "loss":   # per-voxel means of atomically registered pixels
            torch.testing.assert_close(a, b, rtol=1e-2, atol=1e-6, msg=name)
        else:
            assert torch.equal(a.view(torch.int32) if a.dtype == torch.float32 else a,
                               b.view(torch.int32) if b.dtype == torch.float32 else b), name
    assert int((out[0][3] != -float("inf")).sum()) > 1000


# ---- randomised sweep -------------------------------------------------------------------------------------------------

def test_fuzz_slice(cuda_device):
    assert fuzz_run(cases=60, seed0=3, dev=cuda_device) == 0


# ---- the training step ------------------------------------------------------------------------------------------------

DIMS = (32, 32, 32)
W, H = 80, 64


class _Generator(torch.nn.Module):
    """Small seeded stand-in with the reference generator's call signature: Conv3d + BatchNorm3d, and the four dense heads
    as channels of one 19-channel output (the semantic head stays a channel slice of it)."""

    def __init__(self):
        super().__init__()
        self.body = torch.nn.Conv3d(4, 8, 3, padding=1)
        self.bn = torch.nn.BatchNorm3d(8)
        self.head = torch.nn.Conv3d(8, 19, 1)

    def forward(self, inputs, mask, pred_sdf=(True, True), pred_color=True, pred_semantic=True):
        x = torch.relu(self.bn(self.body(inputs)))
        out = self.head(x)
        sdf = inputs[:, :1].to(out.dtype) + 0.3 * torch.tanh(out[:, 1:2])
        return out[:, :1] + 3.0, sdf, torch.tanh(out[:, 2:5]), out[:, 5:19]


def _loss_util():
    return types.SimpleNamespace(
        compute_targets=lambda sdf, truncation, flag, known, colors: (sdf.clone(), colors),
        compute_dense_geo_weights=lambda target, input_occ, truncation, w_surf, w_missing: torch.ones_like(target),
        compute_geo_occ_loss=lambda target, occ, known, weight, truncation: Fn.binary_cross_entropy_with_logits(
            occ, (target.abs() < truncation).float(), weight=weight),
        compute_geo_loss=lambda target, unused, sdf, known, weight, logweight: (weight * (sdf - target).abs()).mean())


class _CopyingGlue:
    """the producer glue as a caller had to use it before: every head through .float().contiguous() first"""

    def __init__(self, sparsify):
        self.sp, self.cache = sparsify, {}

    def _f(self, t):
        if id(t) not in self.cache:
            self.cache[id(t)] = (t, t.float().contiguous())
        return self.cache[id(t)][1]

    def count_locs(self, sdf, truncation, empty=None):
        return self.sp.count_locs(self._f(sdf), truncation, empty)

    def sparsify_predictions(self, sdf, truncation, empty=None, *heads, raycaster=None, counted=None):
        return self.sp.sparsify_predictions(self._f(sdf), truncation, empty, *[self._f(h) for h in heads],
                                            raycaster=raycaster, counted=counted)

    def gather_dense(self, locs, *dense):
        return self.sp.gather_dense(locs, *[self._f(t) for t in dense])


def _sample(device):
    from spsg_b200 import synthetic as S
    sample = S.make_train_sample([0, 1], 1, dims_zyx=DIMS, width=W, height=H,
                                 view_kw=dict(center=(16.0, 16.0, 14.0), radius=38.0, height=30.0))
    sample = {k: torch.from_numpy(v).to(device) for k, v in sample.items()}
    sample["known"] = None
    return sample


def _step(device, model, **kw):
    from spsg_b200 import synthetic as S
    from spsg_b200.train_step import ViewGuidedTrainStep
    cw = torch.tensor(S.CLASS_WEIGHTS, dtype=torch.float32, device=device)
    return ViewGuidedTrainStep(model, _loss_util(), 2, DIMS, W, H, cw, max_num_locs_per_sample=int(DIMS[0] * DIMS[1] * DIMS[2]),
                               device=device, **kw)


class _GradOnly:
    def __init__(self, model):
        self.model = model

    def zero_grad(self, set_to_none=True):
        self.model.zero_grad(set_to_none=True)

    def step(self):
        pass


def test_bf16_step_equals_the_copying_route(cuda_device, monkeypatch):
    from spsg_b200 import sparsify, train_step
    torch.manual_seed(1234)
    model = train_step.prepare_generator(_Generator().to(cuda_device))
    sample = _sample(cuda_device)
    seen = {}
    real_sp = sparsify.sparsify_predictions

    def spy(sdf, truncation, empty=None, *heads, **kw):
        if kw.get("counted") is not None:
            seen["heads"] = (sdf.dtype, [(h.dtype, h.stride(1) == 1) for h in heads])
        return real_sp(sdf, truncation, empty, *heads, **kw)

    step = _step(cuda_device, model, autocast_bf16=True)
    monkeypatch.setattr(sparsify, "sparsify_predictions", spy)
    loss = step({k: v for k, v in sample.items()}, optimizer=_GradOnly(model))
    monkeypatch.setattr(sparsify, "sparsify_predictions", real_sp)
    got = torch.cat([q.grad.reshape(-1) for q in model.parameters()])
    assert seen["heads"] == (torch.bfloat16, [(torch.bfloat16, True), (torch.bfloat16, True)])   # in place, NDHWC
    assert step.last["num_locs"] > 1000

    copying = _step(cuda_device, model, autocast_bf16=True)
    monkeypatch.setattr(train_step, "sparsify", _CopyingGlue(sparsify))
    loss_r = copying({k: v for k, v in sample.items()}, optimizer=_GradOnly(model))
    want = torch.cat([q.grad.reshape(-1) for q in model.parameters()])
    assert copying.last["num_locs"] == step.last["num_locs"]
    assert loss.dtype == loss_r.dtype and torch.equal(loss, loss_r), (float(loss), float(loss_r))
    rel = float((got - want).norm() / want.norm())
    assert rel < 1e-3, rel


def test_bf16_step_trains(cuda_device):
    from spsg_b200 import train_step
    torch.manual_seed(4321)
    model = train_step.prepare_generator(_Generator().to(cuda_device))
    sample = _sample(cuda_device)
    step = _step(cuda_device, model, autocast_bf16=True)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    losses = [float(step(sample, optimizer=opt)) for _ in range(6)]
    assert all(torch.isfinite(torch.tensor(losses)))
    assert losses[-1] < losses[0], losses


def test_switch_off_is_the_float32_step(cuda_device):
    """autocast_bf16=False is the float32 step"""
    from spsg_b200 import train_step
    torch.manual_seed(77)
    model = train_step.prepare_generator(_Generator().to(cuda_device))
    sample = _sample(cuda_device)
    a = _step(cuda_device, model)(sample, optimizer=_GradOnly(model))
    b = _step(cuda_device, model, autocast_bf16=False)(sample, optimizer=_GradOnly(model))
    assert a.dtype == torch.float32 and torch.equal(a, b)
