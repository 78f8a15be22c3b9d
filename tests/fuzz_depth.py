"""Randomised check of the depth-frame utilities (not collected by pytest): every case runs the four entry points and
Depth2Normals (both launch forms) against the CPU restatement tests/depth_oracle.py, bit for bit, with the oracle's
exponentials taken from the device.  Where the compiled reference extension (oracle/_ref) is built, Depth2Normals is
also compared with it on the cases the reference defines (every 11x11 window keeps two valid depths: below that it reads
out of bounds; no NaN pixels).
Cases (depth_oracle.random_case): shapes down to 1 x 1, random sigmas for the filter, per-frame intrinsics, -inf / NaN /
+inf / sub-millimetre / negative pixels, windows with fewer than two valid depths, fill budgets 0 to 128.
usage: python tests/fuzz_depth.py [cases] [seed]"""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
from oracle import ref_driver as refdriver
from spsg_b200 import depth_utils_cuda as mine
from spsg_b200.depth_utils import Depth2Normals
from tests import depth_oracle as O

cases = int(sys.argv[1]) if len(sys.argv) > 1 else 100
seed0 = int(sys.argv[2]) if len(sys.argv) > 2 else 0
dev = torch.device("cuda", 0)
e32 = lambda x: torch.exp(torch.from_numpy(np.ascontiguousarray(x, np.float32)).to(dev)).cpu().numpy()
e64 = lambda x: torch.exp(torch.from_numpy(np.ascontiguousarray(x, np.float64)).to(dev)).cpu().numpy()
with_ref = refdriver.depth_available()
bits = lambda t: O.bits(t.detach().cpu().numpy() if isinstance(t, torch.Tensor) else t)
same = lambda a, b: np.array_equal(bits(a), bits(b))
bad = ref_cases = 0
t0 = time.time()
for c in range(cases):
    rng = np.random.default_rng(seed0 * 104729 + c)
    depth, intr, sigma_d, sigma_r, iters = O.random_case(rng)
    b, _, h, w = depth.shape
    d = torch.from_numpy(depth).to(dev)
    k = torch.from_numpy(intr).to(dev)
    wrong = []
    out = torch.zeros_like(d)
    mine.bilateral_filter_floatmap(out, d, sigma_d, sigma_r)
    if not same(out, O.bilateral(depth, sigma_d, sigma_r, e32, e64)):
        wrong.append("bilateral")
    mine.median_fill_depthmap(out, d)
    if not same(out, O.median_fill(depth)):
        wrong.append("median")
    cam = torch.zeros(b, h, w, 3, device=dev)
    mine.convert_depth_to_cameraspace(cam, d, k, 0.0, 0.0)
    want_cam = O.camspace(depth, intr)
    nrm = torch.zeros_like(cam)
    mine.compute_normals(nrm, cam)
    if not same(cam, want_cam) or not same(nrm, O.normals(want_cam)):
        wrong.append("camspace/normals")
    want = O.depth2normals(depth, intr, iters, e32, e64)
    for coop in (True, False):
        if coop:
            os.environ.pop("SPSG_DEPTH_NO_COOPERATIVE", None)
        else:
            os.environ["SPSG_DEPTH_NO_COOPERATIVE"] = "1"
        d_mine = d.clone()
        mod = Depth2Normals(b, w, h, 0.1 / 0.02, 6.0 / 0.02, max_num_fill_iters=iters, device=dev)
        got = mod(d_mine, k)
        ok = (got is None) == want["none"] and same(d_mine, want["depth"]) and same(mod.filter_helper, want["filtered"]) \
            and same(mod.camspace, want["camspace"]) and same(mod.normals, want["normals"]) and \
            np.array_equal(mod.hole_counts.cpu().numpy(), want["hole_counts"])
        if not ok:
            wrong.append("depth2normals" + ("" if coop else " (launch per pass)"))
    os.environ.pop("SPSG_DEPTH_NO_COOPERATIVE", None)
    if with_ref:
        cnt = torch.nn.functional.avg_pool2d(torch.from_numpy(O.valid(depth)).float(), 11, stride=1, padding=5,
                                             divisor_override=1)
        if float(cnt.min()) >= 1.5 and not np.isnan(depth).any():
            ref_cases += 1
            d_ref = d.clone()
            filt, rcam, rnrm = torch.zeros_like(d), torch.zeros(b, h, w, 3, device=dev), torch.zeros(b, h, w, 3, device=dev)
            ref = refdriver.ref_depth2normals(d_ref, k, filt, rcam, rnrm, max_num_fill_iters=iters)
            if (ref is None) != want["none"] or not same(d_ref, want["depth"]) or not same(filt, want["filtered"]) or \
                    (ref is not None and not (same(rcam, want["camspace"]) and same(rnrm, want["normals"]))):
                wrong.append("reference extension")
    if wrong:
        bad += 1
        print("MISMATCH case %d: b %d h %d w %d sigma %g/%g iters %d none %s: %s" % (
            c, b, h, w, sigma_d, sigma_r, iters, want["none"], ", ".join(wrong)), flush=True)
print("%d cases, %d mismatching (oracle%s), %.1f s" % (
    cases, bad, " + reference extension on %d" % ref_cases if with_ref else "", time.time() - t0))
sys.exit(1 if bad else 0)
