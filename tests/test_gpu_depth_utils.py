"""Depth-frame utilities (csrc/spsg_depth.cu behind the C ABI) against the compiled reference depth_utils extension
(oracle/_ref/spsg_ref_depth_utils_cuda.so) on identical synthetic depth frames.  Bar: bit-exact, including the in-place
hole filling of the caller's depth tensor."""
import numpy as np
import pytest
import torch

from oracle import ref_driver as refdriver

pytestmark = pytest.mark.gpu


def _frames(device, batch=3, h=96, w=128, holes=0.03, seed=0, hole_blocks=True):
    g = torch.Generator().manual_seed(seed)
    yy, xx = torch.meshgrid(torch.arange(h, dtype=torch.float32), torch.arange(w, dtype=torch.float32), indexing="ij")
    depth = []
    for b in range(batch):
        d = 1.2 + 0.004 * xx + 0.002 * yy * (b + 1) + 0.15 * torch.sin(xx / 9.0 + b) * torch.cos(yy / 7.0)
        d = d + 0.01 * torch.randn(h, w, generator=g)
        d[torch.rand(h, w, generator=g) < holes] = 0.0
        if hole_blocks:
            d[20 + b:25 + b, 30:36] = 0.0           # a 5x6 hole: needs the 11x11 window
        depth.append(d)
    depth = torch.stack(depth)[:, None].contiguous().to(device)
    intr = torch.tensor([[107.6, 107.7, w / 2 - 0.5, h / 2 - 0.5]] * batch, device=device)
    return depth, intr


def _need_ref():
    if not refdriver.depth_available(pinned=True):
        pytest.skip("oracle/_ref depth_utils not built (run __graft_entry__.build() where /root/reference exists)")


def _bits_equal(a, b):
    return torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def test_individual_entry_points_bit_exact(cuda_device):
    _need_ref()
    from spsg_b200 import depth_utils_cuda as mine
    ref = refdriver.depth_module(pinned=True)
    depth, intr = _frames(cuda_device)
    b, _, h, w = depth.shape
    fa, fb = torch.zeros_like(depth), torch.zeros_like(depth)
    mine.bilateral_filter_floatmap(fa, depth, 2.0, 0.1)
    ref.bilateral_filter_floatmap(fb, depth, 2.0, 0.1)
    assert _bits_equal(fa, fb), "bilateral: %d values differ" % int((fa != fb).sum())
    ma, mb = torch.zeros_like(depth), torch.zeros_like(depth)
    mine.median_fill_depthmap(ma, depth)
    ref.median_fill_depthmap(mb, depth)
    assert _bits_equal(ma, mb), "median fill: %d values differ" % int((ma != mb).sum())
    assert int((depth == 0).sum()) > int((ma == 0).sum())          # holes were filled
    ca, cb = torch.zeros(b, h, w, 3, device=cuda_device), torch.zeros(b, h, w, 3, device=cuda_device)
    mine.convert_depth_to_cameraspace(ca, depth, intr, 0.0, 0.0)
    ref.convert_depth_to_cameraspace(cb, depth, intr, 0.0, 0.0)
    assert _bits_equal(ca, cb)
    na, nb = torch.zeros_like(ca), torch.zeros_like(cb)
    mine.compute_normals(na, ca)
    ref.compute_normals(nb, cb)
    assert _bits_equal(na, nb)


@pytest.mark.parametrize("holes", [0.0, 0.03])
def test_depth2normals_pipeline_bit_exact(cuda_device, holes):
    _need_ref()
    from spsg_b200.depth_utils import Depth2Normals
    depth, intr = _frames(cuda_device, holes=holes, hole_blocks=holes > 0, seed=4)
    b, _, h, w = depth.shape
    d_mine, d_ref = depth.clone(), depth.clone()
    mod = Depth2Normals(b, w, h, 0.1 / 0.02, 6.0 / 0.02, device=cuda_device)
    got = mod(d_mine, intr)
    filt, cam, nrm = torch.zeros_like(depth), torch.zeros(b, h, w, 3, device=cuda_device), torch.zeros(b, h, w, 3, device=cuda_device)
    want = refdriver.ref_depth2normals(d_ref, intr, filt, cam, nrm, pinned=True)
    assert (got is None) == (want is None)
    assert got is not None, "the synthetic holes are meant to be fillable"
    assert got.shape == (b, 3, h, w)
    assert _bits_equal(got, want), "normals: %d values differ" % int((got != want).sum())
    assert _bits_equal(d_mine, d_ref), "in-place filled depth differs"
    assert _bits_equal(mod.camspace, cam)
    assert _bits_equal(mod.filter_helper, filt)
    if holes > 0:
        assert not torch.equal(d_mine, depth)       # the caller's frame was modified in place
        assert int((d_mine == 0).sum()) == 0


def test_depth2normals_returns_none_when_holes_remain(cuda_device):
    """A hole wider than the fill rounds can close: Depth2Normals returns None (depth_utils.py:93-95, train.py:537-541).

    Deep inside such a hole the 11x11 window holds fewer than two valid depths, and there the reference kernel indexes
    one element past its sorted array (depth_utils_cuda_kernel.cu:133, `diameter*diameter-numValid+(numValid+1)/2` = 121):
    it fills the pixel with whatever the thread's stack held, so its result depends on the kernels that ran before.  This
    implementation leaves those pixels unfilled (0).  The reference is therefore compared only where it is defined: one
    median pass, pixels whose window holds at least two valid depths."""
    _need_ref()
    from spsg_b200 import depth_utils_cuda as mine
    from spsg_b200.depth_utils import Depth2Normals
    ref = refdriver.depth_module(pinned=True)
    depth, intr = _frames(cuda_device, batch=1, holes=0.0, hole_blocks=False, seed=2)
    depth[:, :, 10:70, 20:100] = 0.0                 # far wider than what one fill round (2 x 5 pixels) can close
    b, _, h, w = depth.shape
    valid_count = torch.nn.functional.avg_pool2d((depth != 0).float(), 11, stride=1, padding=5, divisor_override=1)
    defined = (depth != 0) | (valid_count > 1.5)
    assert int((~defined).sum()) > 0
    ma, mb = torch.zeros_like(depth), torch.zeros_like(depth)
    mine.median_fill_depthmap(ma, depth)
    ref.median_fill_depthmap(mb, depth)
    assert _bits_equal(ma[defined], mb[defined])
    assert bool((ma[~defined] == 0).all())
    d_mine = depth.clone()
    mod = Depth2Normals(b, w, h, 5.0, 300.0, max_num_fill_iters=4, device=cuda_device)
    assert mod(d_mine, intr) is None
    assert int((d_mine == 0).sum()) > 0              # partially filled in place, holes remain
    assert int((d_mine == 0).sum()) < int((depth == 0).sum())


@pytest.mark.parametrize("shape", [(3, 96, 128), (8, 256, 320), (2, 61, 75)])
def test_single_launch_pipeline_equals_launch_per_pass(cuda_device, shape, monkeypatch):
    """The fill rounds + normals of Depth2Normals are one cooperative launch (grid barriers between the passes);
    SPSG_DEPTH_NO_COOPERATIVE selects the
    launch-per-pass form of the same passes.  Same normals, filled depth, helper images and hole counts, bit for bit --
    including frames with more tiles than resident CTAs, ragged tile edges and a hole no round can close."""
    from spsg_b200.depth_utils import Depth2Normals
    b, h, w = shape
    depth, intr = _frames(cuda_device, batch=b, h=h, w=w, holes=0.04, hole_blocks=True, seed=9)
    depth[0, :, 5:50, 8:60] = 0.0                    # frame 0 keeps holes for a few rounds
    results = []
    for no_coop in (False, True):
        if no_coop:
            monkeypatch.setenv("SPSG_DEPTH_NO_COOPERATIVE", "1")
        else:
            monkeypatch.delenv("SPSG_DEPTH_NO_COOPERATIVE", raising=False)
        d = depth.clone()
        mod = Depth2Normals(b, w, h, 5.0, 300.0, device=cuda_device)
        out = mod(d, intr)
        torch.cuda.synchronize()
        results.append((out, d, mod.filter_helper.clone(), mod.camspace.clone(), mod.normals.clone(), mod.hole_counts.clone()))
    one, many = results
    assert (one[0] is None) == (many[0] is None)
    for x, y, name in zip(one[1:], many[1:], ("depth", "filtered", "camspace", "normals", "hole counts")):
        assert torch.equal(x.view(torch.int32) if x.dtype == torch.float32 else x,
                           y.view(torch.int32) if y.dtype == torch.float32 else y), name
