"""Parity of the CUDA path (through the public module / C ABI) against the compiled reference extension
(oracle/_ref, the bit-exact pin) and the CPU oracle, on identical seeded synthetic chunks and camera poses.

Bars (BASELINE.json north_star): hit masks, hit voxel indices and every rendered value bit-exact vs the
reference extension on the same GPU; voxel gradients within 1e-3 relative (the reference accumulates them with
float atomics in arbitrary order)."""
import numpy as np
import pytest
import torch

from oracle import ref_driver as refdriver
from tests.common import bits, count_bit_mismatch, hit_image_from_mapping, scene_tensors, views

pytestmark = pytest.mark.gpu

NINF = -float("inf")


def _mine(device, batch_size, dims, w, h, n_max, dmin=None, dmax=None, thresh=None, inc=None, frames=1, max_pix=64):
    from spsg_b200 import synthetic as S
    from spsg_b200.raycast_rgbd import RaycastRGBD
    return RaycastRGBD(batch_size, dims, w, h, S.DEPTH_MIN if dmin is None else dmin,
                       S.DEPTH_MAX if dmax is None else dmax, S.THRESH_SAMPLE_DIST if thresh is None else thresh,
                       S.RAY_INCREMENT if inc is None else inc, max_num_frames=frames,
                       max_num_locs_per_sample=n_max, max_pixels_per_voxel=max_pix, device=device)


def _ref(device, batch_size, dims, w, h, n_max, dmin=None, dmax=None, thresh=None, inc=None, max_pix=64):
    from spsg_b200 import synthetic as S
    if not refdriver.available(pinned=True):
        pytest.skip("oracle/_ref not built (run __graft_entry__.build() where /root/reference exists)")
    return refdriver.RefRaycaster(batch_size, dims, w, h, S.DEPTH_MIN if dmin is None else dmin,
                                  S.DEPTH_MAX if dmax is None else dmax,
                                  S.THRESH_SAMPLE_DIST if thresh is None else thresh,
                                  S.RAY_INCREMENT if inc is None else inc, n_max, max_pix, device=device, pinned=True)


def _assert_render_equal(mine, ref, what=""):
    names = ("color", "depth", "normal", "semantic")
    for name, a, b in zip(names, mine, ref):
        bad = count_bit_mismatch(a, b)
        assert bad == 0, "%s %s: %d of %d values differ bitwise" % (what, name, bad, a.numel())


@pytest.mark.parametrize("view_seed", [0, 1, 2, 3])
def test_forward_bit_exact_config2(cuda_device, view_seed):
    """BASELINE config 2: one chunk, one 320x256 view, all four outputs."""
    from spsg_b200 import synthetic as S
    batch, t = scene_tensors([view_seed], cuda_device)
    n = t["locs"].shape[0]
    _, _, view, intr = views(1, 1, cuda_device, seed=view_seed)
    mine = _mine(cuda_device, 1, S.DIMS_ZYX, S.WIDTH, S.HEIGHT, n)
    ref = _ref(cuda_device, 1, S.DIMS_ZYX, S.WIDTH, S.HEIGHT, n)
    out_m = mine(t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, intr)
    out_r = ref.forward(t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, intr)
    _assert_render_equal(out_m, out_r)
    hit = out_m[1] != NINF
    assert hit.float().mean().item() > 0.3
    assert torch.equal(mine.sparse_mapping, ref.sparse_mapping)
    assert torch.equal(mine.mapping3dto2d_num[:n], ref.mapping3dto2d_num[:n])
    assert int(ref.mapping3dto2d_num[:n].max().item()) <= 64  # deterministic regime (SURVEY.md section 8(d))
    hm = hit_image_from_mapping(mine.mapping3dto2d, mine.mapping3dto2d_num, t["locs"], 1, S.HEIGHT, S.WIDTH)
    hr = hit_image_from_mapping(ref.mapping3dto2d, ref.mapping3dto2d_num, t["locs"], 1, S.HEIGHT, S.WIDTH)
    assert torch.equal(hm, hr), "hit voxel indices differ"
    assert torch.equal(hm >= 0, hit)


@pytest.mark.parametrize("flags", [1, 2, 3])
def test_skipping_is_observationally_identical(cuda_device, flags):
    """Ray/box clipping and empty-brick skipping (flags switch them off) must not change a single bit."""
    from spsg_b200 import synthetic as S
    batch, t = scene_tensors([5], cuda_device)
    n = t["locs"].shape[0]
    _, _, view, intr = views(1, 1, cuda_device, seed=5)
    a = _mine(cuda_device, 1, S.DIMS_ZYX, S.WIDTH, S.HEIGHT, n)
    b = _mine(cuda_device, 1, S.DIMS_ZYX, S.WIDTH, S.HEIGHT, n)
    b.flags = flags
    out_a = a(t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, intr)
    out_b = b(t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, intr)
    _assert_render_equal(out_a, out_b, "flags=%d" % flags)
    assert torch.equal(a.mapping3dto2d_num[:n], b.mapping3dto2d_num[:n])


@pytest.mark.parametrize("chunks,frames", [(1, 1), (3, 2)])
def test_map_placement_paths_agree_bit_for_bit(cuda_device, chunks, frames):
    """The two homes of the march maps -- TMA-staged shared memory with chunk-bound CTAs (default for one chunk) and L1 with
    one global tile counter (default for several) -- render identical images and register identical pixel counts, and both
    equal the reference."""
    from spsg_b200 import _native as N
    from spsg_b200 import synthetic as S
    w, h = 160, 128
    batch, t = scene_tensors(list(range(30, 30 + chunks)), cuda_device)
    n = t["locs"].shape[0]
    _, _, view, intr = views(chunks, frames, cuda_device, seed=6, width=w, height=h)
    outs, nums = [], []
    for flag in (N.SPSG_FLAG_SMEM_MAPS, N.SPSG_FLAG_GLOBAL_MAPS):
        m = _mine(cuda_device, chunks, S.DIMS_ZYX, w, h, n, frames=frames)
        m.flags = flag
        outs.append([o.clone() for o in m(t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, intr)])
        nums.append(m.mapping3dto2d_num[:n * frames].clone())
    _assert_render_equal(outs[0], outs[1], "smem vs global maps")
    assert torch.equal(nums[0], nums[1])
    ref = _ref(cuda_device, chunks, S.DIMS_ZYX, w, h, n)
    for f in range(frames):
        sel = torch.arange(chunks, device=cuda_device) * frames + f
        out_r = ref.forward(t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view[sel].contiguous(), intr[sel].contiguous())
        for a, b in zip(outs[1], out_r):
            assert count_bit_mismatch(a[sel], b) == 0


@pytest.mark.parametrize("inc,dmin,thresh", [(0.3, 5.0, None), (1.7, 0.0, None), (0.123, 20.0, None),
                                             (0.75, 5.0, None), (0.9, 5.0, 1.5), (1.0, 3.0, 0.4)])
def test_forward_bit_exact_march_parameters(cuda_device, inc, dmin, thresh):
    """Other increments (exact-tie and non-tie roundings of the running sum), depth_min = 0, and thresholds
    small enough that the reference's threshSampleDist tests reject crossings (kernel.cu:211-213)."""
    from spsg_b200 import synthetic as S
    w, h = 160, 128
    batch, t = scene_tensors([11], cuda_device)
    n = t["locs"].shape[0]
    _, _, view, intr = views(1, 1, cuda_device, seed=7, width=w, height=h)
    mine = _mine(cuda_device, 1, S.DIMS_ZYX, w, h, n, dmin=dmin, inc=inc, thresh=thresh)
    ref = _ref(cuda_device, 1, S.DIMS_ZYX, w, h, n, dmin=dmin, inc=inc, thresh=thresh)
    out_m = mine(t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, intr)
    out_r = ref.forward(t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, intr)
    _assert_render_equal(out_m, out_r, "inc=%g" % inc)
    assert torch.equal(mine.mapping3dto2d_num[:n], ref.mapping3dto2d_num[:n])


def test_forward_bit_exact_batch_and_odd_sizes(cuda_device):
    """Two different chunks in one call, image size not a multiple of the CTA tile, camera inside the chunk,
    axis-parallel viewing direction, zero normals (kernel.cu:220 keeps -inf)."""
    from spsg_b200 import synthetic as S
    w, h = 93, 71
    batch, t = scene_tensors([2, 3], cuda_device)
    n = t["locs"].shape[0]
    normal = t["normal"].clone()
    normal[::3] = 0.0
    view = np.stack([S.look_at((30.0, 28.0, 60.0), (30.0, 28.0, 0.0), up=(0.0, 1.0, 0.0)),   # inside, looking down -z
                     S.look_at((32.0, -40.0, 40.0), (32.0, 32.0, 40.0))]).astype(np.float32)  # along +y exactly
    intr = np.tile(np.array([[80.0, 80.5, 46.0, 35.0]], np.float32), (2, 1))
    view_t, intr_t = torch.from_numpy(view).to(cuda_device), torch.from_numpy(intr).to(cuda_device)
    mine = _mine(cuda_device, 2, S.DIMS_ZYX, w, h, n)
    ref = _ref(cuda_device, 2, S.DIMS_ZYX, w, h, n)
    out_m = mine(t["locs"], t["sdf"], t["color"], normal, t["semantic"], view_t, intr_t)
    out_r = ref.forward(t["locs"], t["sdf"], t["color"], normal, t["semantic"], view_t, intr_t)
    _assert_render_equal(out_m, out_r)
    hit = out_m[1] != NINF
    assert hit[0].any() and hit[1].any()
    assert ((out_m[2][..., 0] == NINF) & hit).any(), "expected some hit pixels with a zero (unwritten) normal"
    assert torch.equal(mine.mapping3dto2d_num[:n], ref.mapping3dto2d_num[:n])


def test_backward_matches_reference(cuda_device):
    """Voxel gradients for random upstream gradients: within 1e-3 relative of the reference's atomics."""
    from spsg_b200 import synthetic as S
    torch.manual_seed(0)
    batch, t = scene_tensors([4, 6], cuda_device)
    n = t["locs"].shape[0]
    _, _, view, intr = views(2, 1, cuda_device, seed=4)
    mine = _mine(cuda_device, 2, S.DIMS_ZYX, S.WIDTH, S.HEIGHT, n)
    ref = _ref(cuda_device, 2, S.DIMS_ZYX, S.WIDTH, S.HEIGHT, n)
    sdf = t["sdf"].clone().requires_grad_(True)
    col = t["color"].clone().requires_grad_(True)
    nrm = t["normal"].clone().requires_grad_(True)
    sem = t["semantic"].clone().requires_grad_(True)
    out_m = mine(t["locs"], sdf, col, nrm, sem, view, intr)
    out_r = ref.forward(t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, intr)
    grads = [torch.randn_like(o) for o in out_m]
    torch.autograd.backward(out_m, grads)
    d_ref = ref.backward(*grads)
    got = (col.grad, sdf.grad, nrm.grad, sem.grad)
    for name, g, r in zip(("color", "depth->sdf", "normal", "semantic"), got, d_ref):
        assert g.shape == r.shape
        err = (g - r).abs()
        tol = 1e-3 * r.abs() + 1e-5
        assert bool((err <= tol).all()), "%s grads: max err %g" % (name, err.max().item())
    hit_voxels = ref.mapping3dto2d_num[:n] > 0
    assert bool((sdf.grad[~hit_voxels] == 0).all())
    assert hit_voxels.any()


def test_multi_view_equals_looped_reference(cuda_device):
    """F views per chunk in one call == F reference calls (one view each) with gradients accumulated."""
    from spsg_b200 import synthetic as S
    torch.manual_seed(1)
    w, h, F = 160, 128, 3
    batch, t = scene_tensors([8, 9], cuda_device)
    n = t["locs"].shape[0]
    _, _, view, intr = views(2, F, cuda_device, seed=3, width=w, height=h)
    mine = _mine(cuda_device, 2, S.DIMS_ZYX, w, h, n, frames=F)
    ref = _ref(cuda_device, 2, S.DIMS_ZYX, w, h, n)
    sdf = t["sdf"].clone().requires_grad_(True)
    sem = t["semantic"].clone().requires_grad_(True)
    out_m = mine(t["locs"], sdf, t["color"], t["normal"], sem, view, intr)
    assert out_m[1].shape[0] == 2 * F
    grads = [torch.randn_like(o) for o in out_m]
    torch.autograd.backward(out_m, grads)
    acc = [torch.zeros(n, c, device=cuda_device) for c in (3, 1, 3, 14)]
    for f in range(F):
        sel = torch.arange(2, device=cuda_device) * F + f   # image of chunk b, view f
        out_r = ref.forward(t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view[sel].contiguous(),
                            intr[sel].contiguous())
        for a, b in zip(out_m, out_r):
            assert count_bit_mismatch(a[sel], b) == 0
        d = ref.backward(*[g[sel].contiguous() for g in grads])
        for a, x in zip(acc, d):
            a += x
    for g, r in ((sdf.grad, acc[1]), (sem.grad, acc[3])):
        err = (g - r).abs()
        assert bool((err <= 1e-3 * r.abs() + 1e-5).all()), "max err %g" % err.max().item()


def test_raycast_occ_bit_exact(cuda_device):
    from spsg_b200 import synthetic as S
    from spsg_b200.raycast_rgbd import RaycastOcc
    if not refdriver.available(pinned=True):
        pytest.skip("oracle/_ref not built")
    w, h = 160, 128
    sdf, _ = S.sdf_volume(3)
    occ = torch.from_numpy((np.abs(sdf) < 1.0).astype(np.uint8))[None, None].to(cuda_device)
    occ = torch.cat([occ, torch.flip(occ, dims=[4])]).contiguous()
    _, _, view, intr = views(2, 1, cuda_device, seed=9, width=w, height=h)
    mine = RaycastOcc(2, S.DIMS_ZYX, w, h, S.DEPTH_MIN, S.DEPTH_MAX, S.RAY_INCREMENT, device=cuda_device)
    got = mine(occ, view, intr)
    want = torch.zeros_like(got)
    opts = torch.FloatTensor([w, h, S.DEPTH_MIN, S.DEPTH_MAX, S.RAY_INCREMENT, 64, 64, 128])
    refdriver.module(pinned=True).raycast_occ(occ, want, view, intr, opts)
    assert torch.equal(got, want)
    assert 0.2 < got.float().mean().item() < 1.0


def test_cuda_vs_cpu_oracle(cuda_device):
    """Pins the CPU restatement (oracle/raycast_oracle.c) against the GPU path: identical hit masks except rays
    whose crossing sits within fp32 epsilon (1/sqrtf vs rsqrtf), which are counted; values within 1e-4."""
    from oracle import oracle as O
    from spsg_b200 import synthetic as S
    w, h = 160, 128
    batch, t = scene_tensors([12], cuda_device)
    n = t["locs"].shape[0]
    view_np, intr_np, view, intr = views(1, 1, cuda_device, seed=12, width=w, height=h)
    mine = _mine(cuda_device, 1, S.DIMS_ZYX, w, h, n)
    out = [o.cpu().numpy() for o in mine(t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, intr)]
    p = O.make_params(S.DIMS_ZYX, w, h, S.DEPTH_MIN, S.DEPTH_MAX, S.THRESH_SAMPLE_DIST, S.RAY_INCREMENT, 1, 1, 64, n)
    sm = O.build_index(batch["locs"], 1, S.DIMS_ZYX)
    ref = O.raycast_forward(p, sm, batch["sdf"], batch["color"], batch["normal"], batch["semantic"], view_np, intr_np,
                            threads=O.max_threads())
    hit_g, hit_c = np.isfinite(out[1]), np.isfinite(ref["depth"])
    ambiguous = int((hit_g != hit_c).sum())
    assert ambiguous <= 8, "%d eps-ambiguous rays" % ambiguous
    both = hit_g & hit_c
    rel = np.abs(out[1][both] - ref["depth"][both]) / np.abs(ref["depth"][both])
    assert rel.max() < 1e-4
    same_voxel = (out[0][both] == ref["color"][both]).all(axis=-1)
    assert same_voxel.mean() > 0.999


def test_empty_and_error_paths(cuda_device):
    from spsg_b200 import raycast_rgbd_cuda, synthetic as S
    w, h = 64, 48
    mine = _mine(cuda_device, 1, S.DIMS_ZYX, w, h, 1000)
    _, _, view, intr = views(1, 1, cuda_device, width=w, height=h)
    z = lambda *s, **k: torch.zeros(*s, device=cuda_device, **k)
    out = mine(z(0, 4, dtype=torch.long), z(0, 1), z(0, 3), z(0, 3), None, view, intr)
    for o in out:
        assert bool((o == NINF).all())
    with pytest.raises(RuntimeError, match="must be a CUDA tensor"):
        raycast_rgbd_cuda.construct_dense_sparse_mapping(torch.zeros(4, 4, dtype=torch.long), mine.sparse_mapping)
    with pytest.raises(RuntimeError, match="must be contiguous"):
        raycast_rgbd_cuda.construct_dense_sparse_mapping(z(4, 8, dtype=torch.long)[:, ::2], mine.sparse_mapping)


def test_golden_vectors_bit_exact(cuda_device):
    """tests/golden/*.npz: outputs of the reference extension recorded on a B200 (tests/golden/make_golden.py).
    Needs no reference binary at run time."""
    import glob
    import os
    files = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "sphere_*.npz")))
    assert files, "golden vectors missing"
    for f in files:
        g = np.load(f)
        dims = tuple(int(x) for x in g["dims_zyx"])
        h, w = g["depth"].shape[1:]
        n = g["locs"].shape[0]
        mine = _mine(cuda_device, 1, dims, w, h, n, dmin=float(g["depth_min"]), dmax=float(g["depth_max"]),
                     thresh=float(g["thresh"]), inc=float(g["inc"]))
        t = {k: torch.from_numpy(g[k]).to(cuda_device) for k in ("locs", "sdf", "color", "normal", "semantic", "view", "intr")}
        sdf = t["sdf"].clone().requires_grad_(True)
        col = t["color"].clone().requires_grad_(True)
        nrm = t["normal"].clone().requires_grad_(True)
        sem = t["semantic"].clone().requires_grad_(True)
        out = mine(t["locs"], sdf, col, nrm, sem, t["view"], t["intr"])
        want = [torch.from_numpy(g[k]).to(cuda_device) for k in ("color_img", "depth", "normal_img", "semantic_img")]
        _assert_render_equal(out, want, os.path.basename(f))
        assert torch.equal(mine.mapping3dto2d_num[:n].cpu(), torch.from_numpy(g["num"]))
        torch.autograd.backward(out, [torch.from_numpy(g[k]).to(cuda_device) for k in ("g_color", "g_depth", "g_normal", "g_semantic")])
        for got, key in ((col.grad, "d_color"), (sdf.grad, "d_depth"), (nrm.grad, "d_normal"), (sem.grad, "d_semantic")):
            ref = torch.from_numpy(g[key]).to(cuda_device)
            assert bool(((got - ref).abs() <= 1e-3 * ref.abs() + 1e-5).all()), key


def test_forward_bit_exact_whole_room_grid(cuda_device):
    """test_scene.py's use: one whole room (grid far larger than a chunk, so the chunk maps do NOT fit in shared memory
    and the forward takes its global-memory map path + the separate block-map kernel), 480x384 top-down view
    (test_scene.py:89-95, 182-187), grid dims not multiples of the 32-voxel super block."""
    from spsg_b200 import synthetic as S
    dims = (72, 132, 168)
    batch, t = scene_tensors([41], cuda_device, dims_zyx=dims)
    n = t["locs"].shape[0]
    w, h = 480, 384
    # camera above the room centre looking down -z, x right, y flipped (test_scene.py:91-95)
    pose = np.eye(4, dtype=np.float32)
    pose[:3, 0], pose[:3, 1], pose[:3, 2] = (1, 0, 0), (0, -1, 0), (0, 0, -1)
    pose[:3, 3] = (dims[2] // 2, dims[1] // 2, dims[0] * 2)
    view = torch.from_numpy(pose[None]).to(cuda_device)
    intr = torch.tensor([[269.112, 269.297, w // 2, h // 2]], device=cuda_device)
    mine = _mine(cuda_device, 1, dims, w, h, n)
    ref = _ref(cuda_device, 1, dims, w, h, n)
    sdf = t["sdf"].clone().requires_grad_(True)
    sem = t["semantic"].clone().requires_grad_(True)
    out_m = mine(t["locs"], sdf, t["color"], t["normal"], sem, view, intr)
    out_r = ref.forward(t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, intr)
    _assert_render_equal(out_m, out_r, "room")
    assert (out_m[1] != NINF).float().mean().item() > 0.03
    assert torch.equal(mine.mapping3dto2d_num[:n], ref.mapping3dto2d_num[:n])
    grads = [torch.randn_like(o) for o in out_m]
    torch.autograd.backward(out_m, grads)
    d_ref = ref.backward(*grads)
    for g, r in ((sdf.grad, d_ref[1]), (sem.grad, d_ref[3])):
        assert bool(((g - r).abs() <= 1e-3 * r.abs() + 1e-5).all())


def test_crowded_voxels_overflow_max_pixels(cuda_device):
    """Camera a few voxels from a wall: hundreds of pixels land on one voxel, far more than max_pixels_per_voxel.  The
    reference keeps an arbitrary subset of 64 (atomic race), so only what is deterministic is compared with it: images
    and per-voxel pixel counters bit-exact.  The backward is checked against its own definition: the mean over the
    pixels this run registered (kernel.cu:391-419)."""
    from spsg_b200 import synthetic as S
    torch.manual_seed(3)
    w, h, max_pix = 160, 128, 16
    batch, t = scene_tensors([0], cuda_device)
    n = t["locs"].shape[0]
    view_np = S.look_at((48.0, 30.0, 40.0), (57.2, 30.0, 40.0))[None]      # 9 voxels in front of the x wall
    view = torch.from_numpy(view_np).to(cuda_device)
    intr = torch.tensor([[134.5, 134.6, 79.5, 63.5]], device=cuda_device)
    mine = _mine(cuda_device, 1, S.DIMS_ZYX, w, h, n, max_pix=max_pix)
    ref = _ref(cuda_device, 1, S.DIMS_ZYX, w, h, n, max_pix=max_pix)
    sdf = t["sdf"].clone().requires_grad_(True)
    sem = t["semantic"].clone().requires_grad_(True)
    out_m = mine(t["locs"], sdf, t["color"], t["normal"], sem, view, intr)
    out_r = ref.forward(t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, intr)
    _assert_render_equal(out_m, out_r, "crowded")
    num = mine.mapping3dto2d_num[:n]
    assert torch.equal(num, ref.mapping3dto2d_num[:n])
    assert int(num.max()) > 4 * max_pix, "the scene is meant to overflow the per-voxel pixel table"
    grads = [torch.randn_like(o) for o in out_m]
    torch.autograd.backward(out_m, grads)
    # own definition: d[v] = mean over the min(num, max_pix) registered pixels of grad[pixel]
    cnt = num.clamp(max=max_pix)
    rows = torch.nonzero(cnt > 0)[:, 0]
    table = mine.mapping3dto2d[:n][rows].long()                           # (R, max_pix) pixel ids
    valid = torch.arange(max_pix, device=cuda_device)[None, :] < cnt[rows][:, None]
    g_depth = grads[1].reshape(-1)[table.clamp(min=0)] * valid
    want = g_depth.sum(1) / cnt[rows]
    got = sdf.grad[rows, 0]
    assert bool(((got - want).abs() <= 1e-4 * want.abs() + 1e-5).all())
    g_sem = grads[3].reshape(-1, 14)[table.clamp(min=0)] * valid[..., None]
    want_s = g_sem.sum(1) / cnt[rows][:, None]
    assert bool(((sem.grad[rows] - want_s).abs() <= 1e-4 * want_s.abs() + 1e-5).all())
    assert bool((sdf.grad[cnt == 0] == 0).all())


def test_oversize_input_is_truncated_like_the_reference_wrapper(cuda_device, capsys):
    """More voxels than mapping3dto2d has rows: the reference wrapper prints an error and renders the first rows only
    (locs / sdf / colours / normals cut, vals_semantic not: raycast_rgbd.py:16-21)."""
    from spsg_b200 import synthetic as S
    w, h = 96, 80
    batch, t = scene_tensors([9], cuda_device)
    n = t["locs"].shape[0]
    keep = n // 2
    _, _, view, intr = views(1, 1, cuda_device, seed=9, width=w, height=h)
    mine = _mine(cuda_device, 1, S.DIMS_ZYX, w, h, keep)
    ref = _ref(cuda_device, 1, S.DIMS_ZYX, w, h, keep)
    with torch.no_grad():
        out_m = mine(t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, intr)
    assert "ERROR: locs size" in capsys.readouterr().out
    out_r = ref.forward(t["locs"][:keep].contiguous(), t["sdf"][:keep].contiguous(), t["color"][:keep].contiguous(),
                        t["normal"][:keep].contiguous(), t["semantic"], view, intr)
    _assert_render_equal(out_m, out_r, "truncated")
    assert torch.equal(mine.mapping3dto2d_num[:keep], ref.mapping3dto2d_num[:keep])
    assert (out_m[1] != NINF).any()


@pytest.mark.parametrize("frames", [1, 3])
def test_backward_reproduces_bit_for_bit(cuda_device, frames):
    """Repeated forward + backward passes give bit-identical voxel gradients although the order in which warps register a
    voxel's pixels (the rows of mapping3dto2d) and the order of the work list change from run to run -- the gather sums a
    voxel's pixels in double and, with several views per chunk and SPSG_FLAG_DETERMINISTIC_GRADS, its per-view means in view
    order: no float atomics."""
    from spsg_b200 import synthetic as S
    batch, t = scene_tensors([0, 1], cuda_device)
    n = t["locs"].shape[0]
    _, _, view, intr = views(2, frames, cuda_device, seed=0)
    mine = _mine(cuda_device, 2, S.DIMS_ZYX, S.WIDTH, S.HEIGHT, n, frames=frames)
    if frames > 1:
        from spsg_b200 import _native as N
        mine.flags |= N.SPSG_FLAG_DETERMINISTIC_GRADS
    grads, first = None, None
    for rep in range(4):
        leaves = [t[k].clone().requires_grad_(True) for k in ("sdf", "color", "normal", "semantic")]
        out = mine(t["locs"], *leaves, view, intr)
        if grads is None:
            g = torch.Generator(device=cuda_device).manual_seed(1)
            grads = [torch.randn(o.shape, device=cuda_device, generator=g) for o in out]
        torch.autograd.backward(out, grads)
        got = [bits(x.grad).clone() for x in leaves]
        if first is None:
            first = got
        else:
            for name, a, b in zip(("sdf", "color", "normal", "semantic"), first, got):
                assert torch.equal(a, b), "%s gradient changed between runs" % name
