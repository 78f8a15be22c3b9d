"""Randomised parity hunt (run as a script for long hunts; tests/test_gpu_fuzz_slice.py runs a seeded slice under pytest): many random grids / increments / cameras / voxel soups, the CUDA path
against the compiled reference extension, bit for bit.  usage: python tests/fuzz_parity.py [cases] [seed]"""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
from oracle import ref_driver as refdriver
from tests.test_gpu_adversarial import _batch, _cameras
from tests.common import count_bit_mismatch
from spsg_b200.raycast_rgbd import RaycastRGBD

def run(cases=100, seed0=0, dev=None, large=False, pinned=False):
    """Returns the number of mismatching cases."""
    dev = dev or torch.device("cuda", 0)
    assert refdriver.available(pinned), "oracle/_ref not built"
    bad = 0
    t0 = time.time()
    for c in range(cases):
        rng = np.random.default_rng(seed0 * 100003 + c)
        dims = tuple(int(v) for v in rng.integers(3, 70, 3))
        if rng.random() < 0.03:
            dims = tuple(int(v) for v in rng.integers(90, 230, 3))   # too large for the shared-memory maps
        B = int(rng.integers(1, 4))
        kinds = ["noise", "blocky", "special"]
        specs = [(int(rng.integers(0, 1 << 30)), kinds[int(rng.integers(0, 3))]) if rng.random() > 0.1 else None for _ in range(B)]
        if all(s is None for s in specs):
            specs[0] = (1, "noise")
        w, h = int(rng.integers(5, 90)), int(rng.integers(5, 70))
        if large:   # many tiles per SM: the large-launch instantiation of the forward kernel, >1 tile per warp, work stealing
            w, h = int(rng.integers(200, 640)), int(rng.integers(160, 480))
            dims = tuple(int(v) for v in rng.integers(24, 70, 3))
        inc = float(rng.choice([0.9, 0.5, 0.25, 1.0, 0.37, 1.3, 0.123, 2.0, float(rng.uniform(0.05, 2.5))]))
        dmin = float(rng.choice([0.0, 0.0, 5.0, float(rng.uniform(0, 30))]))
        dmax = dmin + float(rng.choice([200.0, 50.0, float(rng.uniform(1, 150))]))
        thresh = float(rng.choice([50.0, 50.0, 1.5, 0.4]))
        max_pix = int(rng.choice([64, 64, 8, 5]))
        t, n = _batch(dims, specs, dev)
        if B * n * max_pix >= (1 << 31) - (1 << 20):
            continue   # the reference indexes mapping3dto2d with 32-bit ints (SURVEY.md section 3.5): it faults beyond 2^31 entries
        view = _cameras(dims, B, int(rng.integers(0, 1 << 30)), dev, lattice=bool(rng.random() < 0.2))
        f = float(rng.uniform(0.4, 1.5)) * w
        intr = torch.tensor([[f, f * float(rng.uniform(0.9, 1.1)), (w - 1) / 2 + float(rng.uniform(-2, 2)), (h - 1) / 2]] * B, device=dev)
        mine = RaycastRGBD(B, dims, w, h, dmin, dmax, thresh, inc, max_num_frames=1, max_num_locs_per_sample=n, max_pixels_per_voxel=max_pix, device=dev)
        ref = refdriver.RefRaycaster(B, dims, w, h, dmin, dmax, thresh, inc, n, max_pix, device=dev, pinned=pinned)
        desc = "case %d: dims %s B %d img %dx%d inc %g dmin %g dmax %g thresh %g max_pix %d specs %s n %d" % (
            c, dims, B, w, h, inc, dmin, dmax, thresh, max_pix, specs, n)
        try:
            with torch.no_grad():
                om = mine(t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, intr)
            torch.cuda.synchronize()
        except Exception as e:
            print("CUDA PATH FAILED", desc, "view", view.tolist(), "intr", intr.tolist(), repr(e)[:200], flush=True); raise
        try:
            orf = ref.forward(t["locs"], t["sdf"], t["color"], t["normal"], t["semantic"], view, intr)
            torch.cuda.synchronize()
        except Exception as e:
            print("REFERENCE FAILED", desc, repr(e)[:200], flush=True); raise
        mism = [count_bit_mismatch(a, b) for a, b in zip(om, orf)]
        same_num = torch.equal(mine.mapping3dto2d_num[:n], ref.mapping3dto2d_num[:n])
        hits = int((om[1] != -float("inf")).sum())
        if any(mism) or not same_num:
            bad += 1
            print("MISMATCH case %d: dims %s B %d img %dx%d inc %g dmin %g dmax %g thresh %g max_pix %d specs %s -> %s num_equal %s hits %d"
                  % (c, dims, B, w, h, inc, dmin, dmax, thresh, max_pix, specs, mism, same_num, hits), flush=True)
    print("%d cases, %d mismatching, %.1f s" % (cases, bad, time.time() - t0))
    return bad


if __name__ == "__main__":
    sys.exit(1 if run(int(sys.argv[1]) if len(sys.argv) > 1 else 100, int(sys.argv[2]) if len(sys.argv) > 2 else 0) else 0)
