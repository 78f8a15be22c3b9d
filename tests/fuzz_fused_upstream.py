"""Randomised check of the fused backward with upstream gradient images (spsg_raycast_backward_loss_upstream; run as a
script for long hunts, tests/test_gpu_fused_upstream.py runs a seeded slice under pytest): random soups, cameras, 1-3 views
per chunk, loss-term switches and random subsets of upstream planes.  After one fused forward, the voxel gradients of
the new entry point must equal spsg_raycast_backward_loss + spsg_raycast_backward of the same images on the same tables,
summed (rtol 1e-5).  usage: python tests/fuzz_fused_upstream.py [cases] [seed]"""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch


def grads_of(m, n):
    return [t[:n].clone() for t in (m.d_depth, m.d_color, m.d_normal, m.d_semantic)]


def upstream_images(images, h, w, planes, gen, dev):
    """Seeded gradient images, (grad_color, grad_depth, grad_normal, grad_semantic); planes not in `planes` are None."""
    shapes = ((images, h, w, 3), (images, h, w), (images, h, w, 3), (images, h, w, 14))
    return tuple((torch.randn(s, generator=gen) * 0.1).to(dev) if k in planes else None for k, s in enumerate(shapes))


def composition(m, p, tg, loss_out, scale, up, n, dims_zyx):
    """(fused + upstream, fused without upstream + plain backward of the same images): the two voxel-gradient lists."""
    from spsg_b200 import losses as L
    from spsg_b200 import raycast_rgbd_cuda as rc
    L.fused_backward(m, p, tg, loss_out, scale, False, upstream=up)
    got = grads_of(m, n)
    L.fused_backward(m, p, tg, loss_out, scale, False)
    want = grads_of(m, n)
    images = p.num_chunks * p.views_per_chunk
    zeros = [torch.zeros_like(b[:images]) for b in (m.image_color, m.image_depth, m.image_normal, m.image_semantic)]
    full = [g if g is not None else z for g, z in zip(up, zeros)]
    rc.backward(full[0], full[1], full[2], full[3], m.sparse_mapping, m.mapping3dto2d, m.mapping3dto2d_num,
                [p.num_chunks, dims_zyx[2], dims_zyx[1], dims_zyx[0], n], m.d_color, m.d_depth, m.d_normal,
                m.d_semantic, views_per_chunk=p.views_per_chunk, workspace_owner=m.workspace, flags=m.flags)
    plain = grads_of(m, n)
    return got, [a + b for a, b in zip(want, plain)]


def close(got, want, rtol=1e-5):
    """Every element within rtol of the reference, plus rtol of the tensor's largest entry for sums that cancel."""
    for a, b in zip(got, want):
        scale = float(b.abs().max()) if b.numel() else 0.0
        if not bool(((a - b).abs() <= rtol * b.abs() + rtol * scale + 1e-12).all()):
            return False
    return True


def run(cases=100, seed0=0, dev=None):
    """Returns the number of mismatching cases."""
    from tests.test_gpu_adversarial import _batch, _cameras
    from spsg_b200 import _native as N
    from spsg_b200 import losses as L
    from spsg_b200.raycast_rgbd import RaycastRGBD
    dev = dev or torch.device("cuda", 0)
    bad = 0
    t0 = time.time()
    for c in range(cases):
        rng = np.random.default_rng(seed0 * 15485863 + c + 7)
        g = torch.Generator().manual_seed(int(rng.integers(0, 1 << 30)))
        dims = tuple(int(v) for v in rng.integers(6, 40, 3))
        B, F = int(rng.integers(1, 4)), int(rng.integers(1, 4))
        kinds = ["noise", "blocky", "special"]
        specs = [(int(rng.integers(0, 1 << 30)), kinds[int(rng.integers(0, 2))]) if rng.random() > 0.15 else None for _ in range(B)]
        if all(s is None for s in specs):
            specs[0] = (3, "blocky")
        w, h = int(rng.integers(8, 70)), int(rng.integers(8, 50))
        t, n = _batch(dims, specs, dev)
        I = B * F
        view = _cameras(dims, I, int(rng.integers(0, 1 << 30)), dev)
        intr = torch.tensor([[float(w), float(w), (w - 1) / 2, (h - 1) / 2]] * I, device=dev)
        rc = RaycastRGBD(B, dims, w, h, 0.0, 150.0, 50.0, float(rng.choice([0.9, 0.5, 1.3])), max_num_frames=F,
                         max_num_locs_per_sample=n, device=dev)
        if F > 1 and rng.random() < 0.5:
            rc.flags = N.SPSG_FLAG_DETERMINISTIC_GRADS
        use_d, use_c, use_s = (bool(rng.random() < 0.7) for _ in range(3))
        images_depth = torch.rand(I, h, w, generator=g) * 2.0
        images_depth[torch.rand(I, h, w, generator=g) < 0.2] = 0.0
        images_color = torch.rand(I, h, w, 3, generator=g)
        label = torch.randint(0, 15, (I, h, w), generator=g).to(torch.uint8)
        wc = (torch.rand(I, h, w, generator=g) + 0.5) if rng.random() < 0.5 else None
        cw = (torch.rand(14, generator=g) + 0.1) if rng.random() < 0.7 else None
        on = lambda use, x: x.to(dev) if (use and x is not None) else None
        targets = (on(use_d, images_depth), on(use_c, images_color), on(use_c, wc), on(use_s, label),
                   None if cw is None else cw.to(dev), 0.02, tuple(float(x) for x in rng.uniform(0.2, 2.0, 3)))
        planes = [k for k in range(4) if rng.random() < 0.6] or [int(rng.integers(0, 4))]
        up = upstream_images(I, h, w, planes, g, dev)
        scale = torch.tensor(float(rng.uniform(0.5, 2.0)), device=dev)
        p, tg, loss_out = L.fused_forward(rc, t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, intr,
                                          targets, False)
        got, want = composition(rc, p, tg, loss_out, scale, up, n, dims)
        if not close(got, want):
            bad += 1
            print("MISMATCH case %d: dims %s B %d F %d img %dx%d terms %s planes %s flags %d" % (
                c, dims, B, F, w, h, (use_d, use_c, use_s), planes, rc.flags), flush=True)
    print("%d cases, %d mismatching, %.1f s" % (cases, bad, time.time() - t0))
    return bad


if __name__ == "__main__":
    sys.exit(1 if run(int(sys.argv[1]) if len(sys.argv) > 1 else 100, int(sys.argv[2]) if len(sys.argv) > 2 else 0) else 0)
