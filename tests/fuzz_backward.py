"""Randomised gradient hunt (run as a script for long hunts; tests/test_gpu_fuzz_slice.py runs a seeded slice under pytest): random soups, cameras and view counts; voxel gradients of the CUDA
path (F views per chunk in one call) against the compiled reference extension (F calls, gradients summed), 1e-3 of the
largest entry.  Cases in which a voxel overflows max_pixels_per_voxel are skipped (the reference keeps an arbitrary subset).
usage: python tests/fuzz_backward.py [cases] [seed]"""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
from oracle import ref_driver as refdriver
from tests.test_gpu_adversarial import _batch, _cameras
from spsg_b200.raycast_rgbd import RaycastRGBD

def run(cases=100, seed0=0, dev=None, pinned=False):
    """Returns the number of mismatching cases."""
    dev = dev or torch.device("cuda", 0)
    assert refdriver.available(pinned), "oracle/_ref not built"
    bad = skipped = 0
    t0 = time.time()
    for c in range(cases):
        rng = np.random.default_rng(seed0 * 100003 + c)
        dims = tuple(int(v) for v in rng.integers(4, 48, 3))
        B, F = int(rng.integers(1, 4)), int(rng.integers(1, 4))
        kinds = ["noise", "blocky", "special"]
        specs = [(int(rng.integers(0, 1 << 30)), kinds[int(rng.integers(0, 3))]) if rng.random() > 0.1 else None for _ in range(B)]
        if all(s is None for s in specs):
            specs[0] = (1, "blocky")
        w, h = int(rng.integers(8, 80)), int(rng.integers(8, 60))
        inc = float(rng.choice([0.9, 0.5, 0.37, 1.3]))
        t, n = _batch(dims, specs, dev)
        view = _cameras(dims, B * F, int(rng.integers(0, 1 << 30)), dev)
        f = float(rng.uniform(0.5, 1.5)) * w
        intr = torch.tensor([[f, f, (w - 1) / 2, (h - 1) / 2]] * (B * F), device=dev)
        mine = RaycastRGBD(B, dims, w, h, 0.0, 150.0, 50.0, inc, max_num_frames=F, max_num_locs_per_sample=n, device=dev)
        ref = refdriver.RefRaycaster(B, dims, w, h, 0.0, 150.0, 50.0, inc, n, 64, device=dev, pinned=pinned)
        leaves = [t[k].clone().requires_grad_(True) for k in ("sdf", "color", "normal", "semantic")]
        out = mine(t["locs"], leaves[0], leaves[1], leaves[2], leaves[3], view, intr)
        g = torch.Generator(device=dev).manual_seed(c)
        grads = [torch.randn(o.shape, device=dev, generator=g) for o in out]
        torch.autograd.backward(out, grads)
        want = [torch.zeros_like(x) for x in leaves]
        overflow = False
        for fv in range(F):
            sel = torch.arange(B, device=dev) * F + fv
            ref.forward(t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view[sel].contiguous(), intr[sel].contiguous())
            overflow |= int(ref.mapping3dto2d_num[:n].max()) > 64
            d_color, d_depth, d_normal, d_sem = ref.backward(*[gr[sel].contiguous() for gr in grads])
            for acc, d in zip(want, (d_depth, d_color, d_normal, d_sem)):
                acc += d
        if overflow:
            skipped += 1
            continue
        for name, a, b in zip(("sdf", "color", "normal", "semantic"), [x.grad for x in leaves], want):
            scale = float(b.abs().max()) + 1e-12
            err = float((a - b).abs().max())
            if not err <= 1e-3 * scale:
                bad += 1
                print("MISMATCH case %d %s: err %.3g scale %.3g dims %s B %d F %d img %dx%d inc %g" % (c, name, err, scale, dims, B, F, w, h, inc), flush=True)
                break
    print("%d cases, %d skipped (pixel-table overflow), %d mismatching, %.1f s" % (cases, skipped, bad, time.time() - t0))
    return bad


if __name__ == "__main__":
    sys.exit(1 if run(int(sys.argv[1]) if len(sys.argv) > 1 else 100, int(sys.argv[2]) if len(sys.argv) > 2 else 0) else 0)
