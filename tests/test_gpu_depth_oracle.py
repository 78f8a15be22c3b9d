"""Depth-frame utilities (csrc/spsg_depth.cu) against the CPU restatement tests/depth_oracle.py, bit for bit, at shapes,
sigmas, windows, intrinsics and fill budgets the recorded reference outputs never saw.  The oracle takes its two
exponentials from the device (``torch.exp`` on CUDA float32 / float64 tensors, libdevice's ``expf`` / ``exp`` like the
kernel: the package is built without fast math); everything else is its own numpy arithmetic.  It is anchored first:
with those exponentials it reproduces every recorded reference output of tests/test_gpu_depth_utils.py.

Every comparison covers every output: the in-place depth, the filter helper, camera space, normals, hole counts and the
None decision of ``Depth2Normals``, in both of its forms (one cooperative launch, and launch per pass).  NaN outputs are
compared as NaN (depth_oracle.bits)."""
import numpy as np
import pytest
import torch

from oracle import ref_driver, ref_pins
from tests import depth_oracle as O
from tests.test_gpu_depth_utils import _frames

pytestmark = pytest.mark.gpu

F32 = np.float32


@pytest.fixture(scope="module")
def dev_exp(cuda_device):
    def e32(x):
        return torch.exp(torch.from_numpy(np.ascontiguousarray(x, F32)).to(cuda_device)).cpu().numpy()

    def e64(x):
        return torch.exp(torch.from_numpy(np.ascontiguousarray(x, np.float64)).to(cuda_device)).cpu().numpy()
    return e32, e64


def _same(got, want, what):
    got = got.detach().cpu().numpy() if isinstance(got, torch.Tensor) else np.asarray(got)
    want = np.asarray(want)
    assert got.shape == want.shape, "%s: shape %s, oracle %s" % (what, got.shape, want.shape)
    if want.dtype == F32:
        bad = O.bits(got) != O.bits(want)
    else:
        bad = got != want
    assert not bad.any(), "%s: %d of %d values differ from the oracle, first at %s (got %r, oracle %r)" % (
        what, int(bad.sum()), bad.size, np.argwhere(bad)[0].tolist(), got[bad][0], want[bad][0])


# --- anchor: the recorded reference outputs ----------------------------------------------------------------------------

class _Counting(O.Module):
    calls = 0

    def __getattribute__(self, name):
        if name in ref_pins.SIGNATURES["depth"]:
            _Counting.calls += 1
        return object.__getattribute__(self, name)


def test_oracle_reproduces_recorded_outputs_with_device_exponentials(dev_exp, monkeypatch):
    """Every depth call test_gpu_depth_utils.py makes through the recorded stand-in, replayed on the oracle: the direct
    bilateral / median / camera-space / normals calls, the median call of the unfillable-hole test and both
    Depth2Normals pipelines (bilateral, fill rounds, camera space, normals).  A call whose key is missing from the table
    had an input that differed, i.e. an upstream output did: a failure."""
    assert ref_pins.recorded()
    impl = _Counting(*dev_exp)
    m = ref_pins.PinnedModule(impl, "depth")
    _Counting.calls = 0
    depth, intr = _frames("cpu")
    b, _, h, w = depth.shape
    m.bilateral_filter_floatmap(torch.zeros_like(depth), depth, 2.0, 0.1)
    m.median_fill_depthmap(torch.zeros_like(depth), depth)
    cam = torch.zeros(b, h, w, 3)
    m.convert_depth_to_cameraspace(cam, depth, intr, 0.0, 0.0)
    m.compute_normals(torch.zeros_like(cam), cam)
    d1, _ = _frames("cpu", batch=1, holes=0.0, hole_blocks=False, seed=2)
    d1[:, :, 10:70, 20:100] = 0.0
    m.median_fill_depthmap(torch.zeros_like(d1), d1)
    monkeypatch.setattr(ref_driver, "depth_module", lambda pinned=False: m)
    for holes in (0.0, 0.03):
        d, k = _frames("cpu", holes=holes, hole_blocks=holes > 0, seed=4)
        out = ref_driver.ref_depth2normals(d, k, torch.zeros_like(d), torch.zeros(b, h, w, 3), torch.zeros(b, h, w, 3),
                                           pinned=True)
        assert out is not None and int((d == 0).sum()) == 0
    assert _Counting.calls == 13      # 5 direct; 3 + 5 of the pipelines (the one with holes fills in one round)


# --- the kernels against the oracle ------------------------------------------------------------------------------------

def _pipeline(depth, intr, iters, dev, monkeypatch, coop):
    from spsg_b200.depth_utils import Depth2Normals
    if coop:
        monkeypatch.delenv("SPSG_DEPTH_NO_COOPERATIVE", raising=False)
    else:
        monkeypatch.setenv("SPSG_DEPTH_NO_COOPERATIVE", "1")
    b, _, h, w = depth.shape
    d = torch.from_numpy(depth).to(dev)
    mod = Depth2Normals(b, w, h, 5.0, 300.0, max_num_fill_iters=iters, device=dev)
    out = mod(d, torch.from_numpy(np.ascontiguousarray(intr)).to(dev))
    torch.cuda.synchronize()
    return out, d, mod


def check_pipeline(depth, intr, iters, dev, exps, monkeypatch):
    """Depth2Normals in both forms against depth_oracle.depth2normals; returns the oracle's result."""
    want = O.depth2normals(depth, intr, iters, *exps)
    for coop in (True, False):
        form = "cooperative" if coop else "launch per pass"
        out, d, mod = _pipeline(depth, intr, iters, dev, monkeypatch, coop)
        assert (out is None) == want["none"], "%s: None decision differs (hole counts %s)" % (form, want["hole_counts"])
        _same(d, want["depth"], form + ": in-place depth")
        _same(mod.filter_helper, want["filtered"], form + ": filter helper")
        _same(mod.camspace, want["camspace"], form + ": camera space")
        _same(mod.normals, want["normals"], form + ": normals")
        _same(mod.hole_counts, want["hole_counts"], form + ": hole counts")
        if out is not None:
            _same(out, want["normals"].transpose(0, 3, 1, 2), form + ": returned normals")
    return want


def check_entry_points(depth, intr, dev, exps, sigma_d=2.0, sigma_r=0.1):
    """The four entry points of depth_utils_cuda against the oracle."""
    from spsg_b200 import depth_utils_cuda as mine
    b, _, h, w = depth.shape
    d = torch.from_numpy(depth).to(dev)
    out = torch.zeros_like(d)
    mine.bilateral_filter_floatmap(out, d, sigma_d, sigma_r)
    _same(out, O.bilateral(depth, sigma_d, sigma_r, *exps), "bilateral (%g, %g)" % (sigma_d, sigma_r))
    mine.median_fill_depthmap(out, d)
    _same(out, O.median_fill(depth), "median fill")
    cam = torch.zeros(b, h, w, 3, device=dev)
    mine.convert_depth_to_cameraspace(cam, d, torch.from_numpy(np.ascontiguousarray(intr)).to(dev), 0.0, 0.0)
    want_cam = O.camspace(depth, intr)
    _same(cam, want_cam, "camera space")
    nrm = torch.zeros_like(cam)
    mine.compute_normals(nrm, cam)
    _same(nrm, O.normals(want_cam), "normals")


SHAPES = [(1, 1, 1), (1, 7, 31), (2, 8, 32), (3, 9, 33), (1, 61, 75), (8, 256, 320), (2, 480, 640)]


@pytest.mark.parametrize("shape", SHAPES, ids=["%dx%dx%d" % s for s in SHAPES])
def test_shapes(cuda_device, dev_exp, monkeypatch, shape):
    """Frames narrower than a 32-pixel tile or shorter than an 8-row one, ragged tile edges, and batches with more tiles
    than the cooperative kernel has resident CTAs (the last two)."""
    b, h, w = shape
    rng = np.random.default_rng(sum(shape))
    depth = O.random_frames(rng, b, h, w, holes=0.04, specials=False)
    depth[0, 0, h // 4:h // 4 + 30, w // 5:w // 5 + 40] = 0.0           # a hole that takes several rounds
    intr = O.random_intrinsics(rng, b, h, w)
    want = check_pipeline(depth, intr, 40, cuda_device, dev_exp, monkeypatch)
    check_entry_points(depth, intr, cuda_device, dev_exp)
    if h * w > 1000:
        assert want["hole_counts"][1] > 0                                    # the big hole needed more than one round


@pytest.mark.parametrize("sigma_r", [0.01, 0.1, 1.0])
@pytest.mark.parametrize("sigma_d", [0.3, 2.0, 2.3, 4.0, 4.01, 5.0])
def test_bilateral_sigmas(cuda_device, dev_exp, sigma_d, sigma_r):
    """Radii 1 to 10: odd radii from fractional sigmas, 8 = ceil(2 * 4.0) the largest with the tabled spatial Gaussian,
    9 = ceil(2 * 4.01) the first computed per tap.  The frames carry -inf, NaN and +inf pixels."""
    from spsg_b200 import depth_utils_cuda as mine
    rng = np.random.default_rng(11)
    depth = O.random_frames(rng, 2, 37, 45, holes=0.1, specials=False)
    flat = depth.reshape(-1)
    pick = rng.choice(flat.size, 33, replace=False)
    flat[pick[:30]], flat[pick[30:32]], flat[pick[32]] = -np.inf, np.nan, np.inf
    d = torch.from_numpy(depth).to(cuda_device)
    out = torch.zeros_like(d)
    mine.bilateral_filter_floatmap(out, d, sigma_d, sigma_r)
    want = O.bilateral(depth, sigma_d, sigma_r, *dev_exp)
    _same(out, want, "bilateral (%g, %g)" % (sigma_d, sigma_r))
    assert np.count_nonzero(np.isfinite(want) & (want != 0)) > depth.size // 4


def _window_frames():
    """One 24 x 40 frame per median-window case (frames are independent, so the cases cannot interact)."""
    h, w = 24, 40
    rng = np.random.default_rng(5)
    f = np.zeros((10, h, w), F32)
    # 0: no valid depth at all (n = 0 everywhere)
    f[1, 12, 20] = 1.5                                                        # 1: n = 1 around one pixel
    f[2, 12, 20], f[2, 14, 23] = 1.5, 2.0                                     # 2: n = 2 and n = 1
    f[3, 12, 20], f[3, 14, 23], f[3, 10, 17] = 1.5, 2.0, 0.7                  # 3: n = 3, 2, 1
    f[4] = 1.75                                                               # 4: all valid values equal
    f[4][rng.random((h, w)) < 0.5] = 0.0
    f[5] = np.exp(rng.uniform(np.log(0.001), np.log(60.0), (h, w)))           # 5: 1 mm to 60 m in one window
    f[5][rng.random((h, w)) < 0.4] = 0.0
    f[6] = rng.choice(np.array([1e-4, 2e-4, -1e-4, -0.5, -3.0, 0.7, 2.0, 0.0], F32), (h, w))   # 6: both sides of 0
    f[7, 5, 5], f[7, 5, 8] = -0.002, 0.004                                    # 7: q = -1 with one other valid depth
    f[7, 15, 30], f[7, 16, 30] = -0.0015, -0.0024                             #    and two q = -1 entries alone
    f[8] = rng.uniform(0.5, 3.0, (h, w))                                      # 8: -inf and NaN pixels
    f[8][rng.random((h, w)) < 0.2] = -np.inf
    f[8][rng.random((h, w)) < 0.05] = np.nan
    f[8][rng.random((h, w)) < 0.2] = 0.0
    f[9] = rng.uniform(0.5, 3.0, (h, w))                                      # 9: holes on every border and corner
    f[9][:2], f[9][-1], f[9][:, :3], f[9][:, -2:] = 0.0, 0.0, 0.0, 0.0
    f[9][5:9, 10:14] = 0.0
    return f[:, None]


def test_median_windows(cuda_device, dev_exp, monkeypatch):
    """Windows with 0, 1, 2 and 3 valid values, all equal (no bit to vote on), spanning 1 mm to 60 m (more than ten
    bits), straddling the sign bit (valid depths of 0.1 mm and negative ones), q = -1 entries, -inf and NaN pixels, and
    holes on every border and corner: the median fill entry point, and the pipeline over the same frames."""
    from spsg_b200 import depth_utils_cuda as mine
    depth = _window_frames()
    d = torch.from_numpy(depth).to(cuda_device)
    out = torch.zeros_like(d)
    mine.median_fill_depthmap(out, d)
    want = O.median_fill(depth)
    _same(out, want, "median fill")
    got = out.cpu().numpy()[:, 0]
    # the documented rule, independently of the oracle: the ((n+1)/2)-th smallest of the n valid quantised depths
    assert not got[0].any() and np.count_nonzero(got[1]) == 1                 # n = 0 and n = 1 leave holes
    assert got[2, 12, 18] == F32(0.001) * F32(2000)                           # {1500, 2000}: the larger
    assert got[3, 12, 18] == F32(0.001) * F32(2000)                           # {700, 1500, 2000}: the largest
    assert got[7, 5, 6] == F32(0.001) * F32(4)                                # {-1, 4}: the q = -1 entry counts
    assert got[7, 15, 31] == 0 and got[7, 15, 30] == F32(-0.0015)             # {-1, -1}: 0; valid pixel copied
    assert np.isnan(got[8]).any() and not np.isneginf(got[8]).any()           # NaN copied, -inf filled or zeroed
    intr = O.random_intrinsics(np.random.default_rng(6), depth.shape[0], 24, 40)
    check_entry_points(depth, intr, cuda_device, dev_exp)
    check_pipeline(depth, intr, 40, cuda_device, dev_exp, monkeypatch)


def test_intrinsics_per_frame(cuda_device, dev_exp, monkeypatch):
    """Every frame its own fx, fy, mx, my: a pass that read one frame's intrinsics for all would differ."""
    rng = np.random.default_rng(21)
    depth = O.random_frames(rng, 4, 30, 50, holes=0.02, specials=False)
    intr = O.random_intrinsics(rng, 4, 30, 50)
    assert not np.array_equal(O.camspace(depth, intr)[1:], O.camspace(depth, np.repeat(intr[:1], 4, 0))[1:])
    check_entry_points(depth, intr, cuda_device, dev_exp)
    check_pipeline(depth, intr, 40, cuda_device, dev_exp, monkeypatch)


@pytest.mark.parametrize("iters", [0, 1, 2, 3, 40, 128])
def test_fill_budgets(cuda_device, dev_exp, monkeypatch, iters):
    """Budgets of no round (0, 1), one (2, 3), twenty and the limit of 64 rounds.  Frame 1 has no valid depth: no budget
    closes it, so every budget above 0 returns None, and frame 0's large hole is filled as far as the budget reaches."""
    rng = np.random.default_rng(31)
    depth = O.random_frames(rng, 2, 64, 80, holes=0.03, specials=False)
    depth[0, 0, 10:50, 15:70] = 0.0
    depth[1] = 0.0
    intr = O.random_intrinsics(rng, 2, 64, 80)
    want = check_pipeline(depth, intr, iters, cuda_device, dev_exp, monkeypatch)
    assert want["none"] == (iters > 0)
    if iters >= 2:
        assert want["hole_counts"][1] < want["hole_counts"][0]               # partly filled in place


@pytest.mark.parametrize("chunk", range(4))
def test_randomised_slice(cuda_device, dev_exp, monkeypatch, chunk):
    """60 seeded random cases (tests/fuzz_depth.py's generator): shapes down to 1 x 1, random sigmas for the filter,
    per-frame intrinsics, -inf / NaN / +inf / sub-millimetre / negative pixels, windows with fewer than two valid
    depths, and every fill budget."""
    for c in range(chunk * 15, chunk * 15 + 15):
        depth, intr, sigma_d, sigma_r, iters = O.random_case(np.random.default_rng(1000 + c))
        check_entry_points(depth, intr, cuda_device, dev_exp, sigma_d, sigma_r)
        check_pipeline(depth, intr, iters, cuda_device, dev_exp, monkeypatch)
