"""Randomised backward hunt against the float64 gather oracle (tests/gather_oracle.py); tests/test_gpu_gather_oracle.py
runs a seeded slice under pytest and uses the same case runner.  Each case renders a random soup with the voxel id in the
normal payload and checks:
  * the forward renders bit-identically with flags 0, with NO_CLIP | NO_BRICK_SKIP (the literal march), and with
    SMEM_MAPS against GLOBAL_MAPS;
  * the payload identities and the registration tables (gather_oracle.pixel_map / check_tables);
  * the plain backward (F views, atomics or deterministic), every entry against the oracle, and in some cases the
    backward that clears its own rows, on d_* pre-filled with NaN;
  * the fused 2D-loss backward with random term switches, targets and upstream planes, and its loss values.
usage: python tests/fuzz_gather.py [cases] [seed]"""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
import numpy as np
import torch

from spsg_b200 import _native as N
from tests import gather_oracle as O

NINF = -float("inf")
MAX_PIX = (1, 5, 16, 17, 33, 64)


def scene(dev, dims, specs, n_keep=None):
    """_batch of test_gpu_adversarial with the voxel id in the normal payload; n_keep = the first rows only."""
    from tests.test_gpu_adversarial import _batch
    t, n = _batch(dims, specs, dev)
    if n_keep is not None:
        n = min(n, n_keep)
        t = {k: v[:n].contiguous() for k, v in t.items()}
    t["normal"] = torch.from_numpy(O.voxel_normals(n)).to(dev)
    return t, n


def slab(dev, n, dims=(16, 16, 16)):
    """Exactly n voxels in one chunk: a slab four voxels thick (sdf = z - 7.5, surface inside it) centred on x = y = 8,
    4 x 4 columns for n <= 64, 8 x 8 for more, listed column by column (a prefix of the rows still holds complete cells)
    and extended by single voxels below it; slab_cameras look down on it."""
    a = 4 if n <= 64 else 8
    rows = [(z, 8 - a // 2 + y, 8 - a // 2 + x) for y in range(a) for x in range(a) for z in (6, 7, 8, 9)]
    rows += [(2, y, x) for y in range(16) for x in range(16)]
    locs = np.array(rows[:n], np.int64)
    locs = np.concatenate([locs, np.zeros((n, 1), np.int64)], 1)
    rng = np.random.default_rng(n)
    sdf = (locs[:, :1] - 7.5 + rng.uniform(-0.1, 0.1, (n, 1))).astype(np.float32)
    t = dict(locs=locs, sdf=sdf, color=rng.random((n, 3), dtype=np.float32),
             normal=O.voxel_normals(n), semantic=rng.standard_normal((n, 14)).astype(np.float32))
    return {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in t.items()}, n


def slab_cameras(dev, count, seed=0):
    from spsg_b200 import synthetic as S
    rng = np.random.default_rng(seed)
    mats = [S.look_at((8 + rng.uniform(-2, 2), 8 + rng.uniform(-2, 2), 16 + rng.uniform(0, 4)), (8.0, 8.0, 7.5),
                      up=(0.0, 1.0, 0.0)) for _ in range(count)]
    return torch.from_numpy(np.stack(mats).astype(np.float32)).to(dev)


def raycaster(dev, B, F, dims, w, h, n, dmin=0.0, dmax=150.0, inc=0.9, max_pix=64, deterministic=False, flags=0):
    from spsg_b200.raycast_rgbd import RaycastRGBD
    m = RaycastRGBD(B, dims, w, h, dmin, dmax, 50.0, inc, max_num_frames=F, max_num_locs_per_sample=n // B + 1,
                    max_pixels_per_voxel=max_pix, device=dev)
    m.flags = flags | (N.SPSG_FLAG_DETERMINISTIC_GRADS if deterministic else 0)
    return m


def intrinsics(dev, count, w, h, scale=1.0):
    f = scale * w
    return torch.tensor([[f, f, (w - 1) / 2, (h - 1) / 2]] * count, device=dev)


def upstream_grads(shapes, dev, seed):
    """Log-uniform magnitudes over 1e-6 .. 1e3, mixed signs, fp32."""
    g = torch.Generator().manual_seed(seed)
    out = []
    for s in shapes:
        mag = 10.0 ** (torch.rand(s, generator=g, dtype=torch.float64) * 9 - 6)
        sign = torch.where(torch.rand(s, generator=g) < 0.5, -1.0, 1.0)
        out.append((mag * sign).float().to(dev))
    return out


def _np(x):
    return x.detach().float().cpu().numpy()


def oracle_tables(m, t, n, F, out):
    color, depth, normal, sem = (_np(o) for o in out)
    vox = O.pixel_map(color, depth, normal, sem, _np(t["color"]), _np(t["semantic"]))
    tab = O.check_tables(vox, m.mapping3dto2d.cpu().numpy(), m.mapping3dto2d_num.cpu().numpy(),
                         t["locs"][:, 3].cpu().numpy(), F)
    return tab, (color, depth, normal, sem)


def leaves(t):
    return [t[k].clone().requires_grad_(True) for k in ("sdf", "color", "normal", "semantic")]


def got_grads(ls):
    sdf, col, nrm, sem = (_np(x.grad) if x.grad is not None else np.zeros(x.shape, np.float32) for x in ls)
    return O.route(sem, col, sdf, nrm)


def check_plain(m, t, n, F, view, intr, seed, what=""):
    """Autograd backward of the module with random upstream images against the oracle.  Returns (tables, near-ties)."""
    ls = leaves(t)
    out = m(t["locs"], *ls, view, intr)
    tab, _ = oracle_tables(m, t, n, F, out)
    grads = upstream_grads([o.shape for o in out], m.image_depth.device, seed)
    torch.autograd.backward(out, grads)
    det = bool(m.flags & N.SPSG_FLAG_DETERMINISTIC_GRADS) and F > 1
    g = O.gather(tab, O.plain_pixel_grads(*(_np(x) for x in grads)), deterministic=det)
    ties = O.compare(got_grads(ls), g, what + " plain", exact=det)
    return tab, ties


def check_self_clearing(m, t, n, F, view, intr, seed, what=""):
    """The raw forward / backward with grads_cleared=False on d_* full of NaN: the backward clears the rows itself."""
    from spsg_b200 import raycast_rgbd_cuda as rc
    dims = m.dims3d
    ws = rc.ModuleWorkspace()
    opts = [m.width, m.height, m.depth_min, m.depth_max, m.thresh_sample_dist, m.ray_increment, dims[2], dims[1], dims[0]]
    rc.forward(m.sparse_mapping, t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, m.image_color,
               m.image_depth, m.image_normal, m.image_semantic, m.mapping3dto2d, m.mapping3dto2d_num, intr, opts,
               views_per_chunk=F, flags=m.flags, build_index=True, workspace_owner=ws)
    images = view.shape[0]
    out = (m.image_color[:images], m.image_depth[:images], m.image_normal[:images], m.image_semantic[:images])
    tab, _ = oracle_tables(m, t, n, F, out)
    grads = upstream_grads([o.shape for o in out], view.device, seed)
    for d in (m.d_color, m.d_depth, m.d_normal, m.d_semantic):
        d.fill_(float("nan"))
    rc.backward(*grads, m.sparse_mapping, m.mapping3dto2d, m.mapping3dto2d_num, [m.batch_size, dims[2], dims[1], dims[0], n],
                m.d_color, m.d_depth, m.d_normal, m.d_semantic, views_per_chunk=F, grads_cleared=False,
                workspace_owner=ws, flags=m.flags)
    det = bool(m.flags & N.SPSG_FLAG_DETERMINISTIC_GRADS) and F > 1
    g = O.gather(tab, O.plain_pixel_grads(*(_np(x) for x in grads)), deterministic=det)
    got = O.route(_np(m.d_semantic[:n]), _np(m.d_color[:n]), _np(m.d_depth[:n]), _np(m.d_normal[:n]))
    return O.compare(got, g, what + " self-clearing", exact=det)


def fused_targets(out, rng, dev, terms=(True, True, True), tie_frac=0.1):
    """Random targets for the three terms (None = off): depth with holes and exact ties, colour with exact ties and a
    weight with zeros, labels with 14, class weights with zeros."""
    color, depth, _, sem = (_np(o) for o in out)
    I, H, W = depth.shape
    vs = np.float32(0.02)
    td = tc = wc = lab = cw = None
    if terms[0]:
        td = (rng.random((I, 1, H, W)) * 2.0).astype(np.float32)
        tie = (rng.random((I, 1, H, W)) < tie_frac) & (depth[:, None] != NINF)
        with np.errstate(invalid="ignore", over="ignore"):
            td = np.where(tie, depth[:, None] * vs, td).astype(np.float32)
        td[rng.random(td.shape) < 0.15] = 0.0
    if terms[1]:
        tc = rng.random((I, H, W, 3)).astype(np.float32)
        tie = (rng.random((I, H, W, 1)) < tie_frac) & (color != NINF)
        tc = np.where(tie, color, tc).astype(np.float32)
        wc = (rng.random((I, 1, H, W)) + 0.5).astype(np.float32)
        wc[rng.random(wc.shape) < 0.1] = 0.0
    if terms[2]:
        lab = rng.integers(0, 15, (I, H, W)).astype(np.uint8)
        cw = (rng.random(14) + 0.1).astype(np.float32)
        cw[rng.integers(0, 14, 2)] = 0.0
    to = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    return dict(images_depth=to(td), images_color=to(tc), weight_color=to(wc), target2d_label=to(lab),
                weight_semantic_class=to(cw)), (td, tc, wc, lab, cw)


def check_fused(m, t, n, F, view, intr, seed, terms=(True, True, True), planes=(), grad_scale=1.0,
                route_="autograd", weights=(0.5, 1.5, 0.8), what=""):
    """Fused backward through render_with_2d_losses (route_ 'autograd') or render_loss_and_voxel_grads ('direct').
    planes: which upstream images (0 colour, 1 depth, 2 normal, 3 semantic) feed the objective (autograd only)."""
    from spsg_b200.losses import render_loss_and_voxel_grads, render_with_2d_losses
    dev = view.device
    rng = np.random.default_rng(seed)
    with torch.no_grad():  # a plain render of the same inputs: the targets are built around it (exact ties)
        pre = [o.clone() for o in m(t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, intr)]
    tg, (td, tc, wc, lab, cw) = fused_targets(pre, rng, dev, terms)
    kw = dict(tg, voxelsize=0.02, weight_depth_loss=weights[0], weight_color_loss=weights[1],
              weight_semantic_loss=weights[2])
    ups = None
    if route_ == "direct":
        loss_out, grads = render_loss_and_voxel_grads(m, t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"],
                                                      view, intr, grad_scale=torch.tensor(grad_scale, device=dev), **kw)
        out = (m.image_color[:view.shape[0]], m.image_depth[:view.shape[0]], m.image_normal[:view.shape[0]],
               m.image_semantic[:view.shape[0]])
        tab, (color, depth, normal, sem) = oracle_tables(m, t, n, F, out)
        got = O.route(*(_np(g) for g in (grads[3], grads[1], grads[0], grads[2])))
        vals = _np(loss_out)
    else:
        ls = leaves(t)
        total, termv, out = render_with_2d_losses(m, t["locs"], *ls, view, intr, differentiable_images=bool(planes), **kw)
        tab, (color, depth, normal, sem) = oracle_tables(m, t, n, F, out)
        obj = total * grad_scale
        if planes:
            ug = upstream_grads([o.shape for o in out], dev, seed + 1)
            ups = [_np(ug[k]) if k in planes else None for k in range(4)]
            for k in planes:
                obj = obj + (out[k].masked_fill(out[k] == NINF, 0.0) * ug[k]).sum()
        obj.backward()
        got = got_grads(ls)
        vals = np.concatenate([_np(termv), _np(total).reshape(1)])
    G, mag, bnd, (want_vals, vbound) = O.fused_pixel_grads(
        color, depth, sem, td, tc, wc, lab, cw, 0.02, weights, grad_scale, ups)
    g = O.gather(tab, G, pixel_bound=bnd, mag=mag)
    O.compare(got, g, what + " fused")
    for k in range(4):
        a, b = float(vals[k]), float(want_vals[k])
        assert (np.isnan(a) and np.isnan(b)) or abs(a - b) <= vbound[k], \
            "%s loss value %d: %r vs float64 %r (bound %.3g)" % (what, k, a, b, vbound[k])
    return tab


def check_forward_flags(m, t, view, intr, what=""):
    """Bit-identical renderings and tables with flags 0, the literal march, and shared- vs global-memory maps."""
    saved = m.flags
    res = []
    for fl in (0, N.SPSG_FLAG_NO_CLIP | N.SPSG_FLAG_NO_BRICK_SKIP, N.SPSG_FLAG_SMEM_MAPS, N.SPSG_FLAG_GLOBAL_MAPS):
        m.flags = fl
        with torch.no_grad():
            out = m(t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, intr)
        res.append(([o.clone() for o in out], m.mapping3dto2d_num.clone()))
    m.flags = saved
    base, num0 = res[0]
    for (out, num), name in zip(res[1:], ("literal march", "smem maps", "global maps")):
        for a, b, plane in zip(out, base, ("colour", "depth", "normal", "semantic")):
            assert torch.equal(a.view(torch.int32), b.view(torch.int32)), "%s: %s %s differs from flags 0" % (what, name, plane)
        assert torch.equal(num, num0), "%s: %s registration counts differ" % (what, name)


def draw(rng):
    """One random case (see the module docstring)."""
    big = rng.random() < 0.15
    dims = tuple(int(v) for v in (rng.integers(90, 231, 3) if big else rng.integers(3, 71, 3)))
    B, F = int(rng.integers(1, 4)), int(rng.integers(1, 5))
    kinds = ["noise", "blocky", "special"]
    specs = [(int(rng.integers(0, 1 << 30)), kinds[int(rng.integers(0, 3))]) for _ in range(B)]
    if B > 1 and rng.random() < 0.3:
        specs[int(rng.integers(0, B))] = None
    if big:
        w, h = int(rng.integers(200, 641)), int(rng.integers(8, 71))
    else:
        w, h = int(rng.integers(1, 91)), int(rng.integers(1, 71))
    dmin, dmax = [(0.0, 150.0), (0.0, 150.0), (80.0, 20.0), (0.0, 0.5), (5.0, 60.0)][int(rng.integers(0, 5))]
    if big:  # one chunk, its first 200 000 rows: the grid takes the global-memory map path, the oracle stays small
        B, specs = 1, specs[:1] if specs[0] is not None else [(1, "blocky")]
    return dict(dims=dims, B=B, F=F, specs=specs, keep=200000 if big else None, w=w, h=h, inc=float(rng.choice([0.9, 0.5, 0.37, 1.3])), dmin=dmin,
                dmax=dmax, max_pix=int(rng.choice(MAX_PIX)), det=bool(rng.random() < 0.5),
                focal=float(rng.uniform(0.5, 1.5)), cam_seed=int(rng.integers(0, 1 << 30)),
                self_clear=bool(rng.random() < 0.3), terms=tuple(bool(x) for x in rng.random(3) < 0.6),
                planes=tuple(int(k) for k in np.nonzero(rng.random(4) < 0.4)[0]),
                grad_scale=float(np.float32(rng.choice([1.0, 0.37, 3.0]))))


def run_case(c, dev, seed):
    from tests.test_gpu_adversarial import _cameras
    t, n = scene(dev, c["dims"], c["specs"], c["keep"])
    B, F = c["B"], c["F"]
    view = _cameras(c["dims"], B * F, c["cam_seed"], dev)
    intr = intrinsics(dev, B * F, c["w"], c["h"], c["focal"])
    m = raycaster(dev, B, F, c["dims"], c["w"], c["h"], n, c["dmin"], c["dmax"], c["inc"], c["max_pix"], c["det"])
    what = "case %s" % {k: v for k, v in c.items() if k != "specs"}
    check_forward_flags(m, t, view, intr, what)
    tab, ties = check_plain(m, t, n, F, view, intr, seed, what)
    if c["self_clear"]:
        ties += check_self_clearing(m, t, n, F, view, intr, seed, what)
    if any(c["terms"]) or c["planes"]:
        check_fused(m, t, n, F, view, intr, seed, c["terms"], c["planes"], c["grad_scale"], what=what)
    return tab.overflow.size > 0, ties


def run(cases=100, seed0=0, dev=None):
    """Returns the number of mismatching cases."""
    dev = dev or torch.device("cuda", 0)
    bad = overflow = ties = 0
    t0 = time.time()
    for k in range(cases):
        rng = np.random.default_rng(seed0 * 100003 + k)
        c = draw(rng)
        try:
            ov, ti = run_case(c, dev, seed0 * 100003 + k)
            overflow += ov
            ties += ti
        except AssertionError as e:
            bad += 1
            print("MISMATCH case %d: %s" % (k, e), flush=True)
    print("%d cases, %d with a pixel-table overflow, %d near-tie entries excluded, %d mismatching, %.1f s"
          % (cases, overflow, ties, bad, time.time() - t0))
    return bad


if __name__ == "__main__":
    sys.exit(1 if run(int(sys.argv[1]) if len(sys.argv) > 1 else 100, int(sys.argv[2]) if len(sys.argv) > 2 else 0) else 0)
