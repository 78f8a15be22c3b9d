#!/usr/bin/env python
"""A/B of the fused backward gather: the library of an earlier revision against the current one, on bench.py's C3 inputs
(8 chunks x 5 views, 320x256, seeded synthetic, all three 2D loss terms), in one call on one GPU.

    python tools/gather_ab.py --build-parent REV      # compile REV's csrc/ + include/ to build/ab_parent/ (no GPU needed)
    python tools/gather_ab.py [--out DIR] [--rounds 3] [--min-window-s 0.5]

Each measurement runs in its own subprocess with SPSG_RAYCAST_LIB selecting the library (the Python package is the
current one for both), the two arms alternated.

Results, parent vs current:
  det_f5, det_f1, det_f5_upstream   SPSG_FLAG_DETERMINISTIC_GRADS at F = 5 (and with seeded colour + semantic upstream
                                    images), one view per chunk at F = 1: d_sdf, d_color, d_normal, d_semantic and loss_out
                                    bit for bit.  Entries one ulp apart are counted separately as exact ties of the
                                    double-precision sum (none are expected: both builds sum the same fp32 terms in the
                                    same order).
  atomic_f5                         the default float atomics: each build adds the same per-view means in whatever order
                                    the atomics land, so the two may differ by 2 (F-1) 2^-24 sum_f |mean_f| per entry
                                    (the gather oracle's multi-view bound, once per build); sum_f |mean_f| is bounded by
                                    the plain gather of the absolute per-pixel loss gradients.
Timing, median over --rounds windows per arm, each >= --min-window-s:
  gather_us   the fused gather kernel, CUDA events of the spsg_timing_* hook (slot 1) over eager steps
  step_ms     bench.py's headline step (fused forward + backward) replayed from a CUDA graph over rotated input sets that
              together exceed the 126 MB L2
The device name and power limit are read in the same call.  Exit status 1 if a result check fails.
"""
import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PKG = "self-supervised-scene-generation-with-semantic-segmentation_b200"
PARENT_LIB = os.path.join(ROOT, "build", "ab_parent", "libspsg_raycast.so")
CURRENT_LIB = os.path.join(ROOT, PKG, "lib", "libspsg_raycast.so")
B, F = 8, 5
CHECKS = ("det_f5", "det_f1", "det_f5_upstream", "atomic_f5")


def build_parent(rev):
    import __graft_entry__ as G
    tmp = tempfile.mkdtemp()
    try:
        tar = subprocess.run(["git", "-C", ROOT, "archive", rev, PKG + "/csrc", "include"], check=True,
                             capture_output=True).stdout
        subprocess.run(["tar", "-x", "-C", tmp], input=tar, check=True)
        csrc = os.path.join(tmp, PKG, "csrc")
        sources = [os.path.join(csrc, f) for f in sorted(os.listdir(csrc)) if f.endswith(".cu")]
        flags = [f if f != os.path.join(ROOT, "include") else os.path.join(tmp, "include") for f in G.NVCC_FLAGS]
        os.makedirs(os.path.dirname(PARENT_LIB), exist_ok=True)
        subprocess.run([G.NVCC] + flags + sources + ["-o", PARENT_LIB], check=True)
    finally:
        shutil.rmtree(tmp)
    with open(os.path.join(os.path.dirname(PARENT_LIB), "REVISION"), "w") as f:
        f.write(subprocess.run(["git", "-C", ROOT, "rev-parse", rev], check=True, capture_output=True,
                               text=True).stdout)
    print("built", PARENT_LIB, "from", rev)


# ---------------------------------------------------------------------------------------------------------------------
# workers (one library each, selected by SPSG_RAYCAST_LIB)
# ---------------------------------------------------------------------------------------------------------------------

def _inputs(dev, views):
    import bench
    from spsg_b200 import synthetic as S
    from spsg_b200.raycast_rgbd import RaycastRGBD
    d = {k: v.to(dev) for k, v in bench.make_host_sets(1, B, views, 0)[0].items()}
    m = RaycastRGBD(B, S.DIMS_ZYX, S.WIDTH, S.HEIGHT, S.DEPTH_MIN, S.DEPTH_MAX, S.THRESH_SAMPLE_DIST, S.RAY_INCREMENT,
                    max_num_frames=views, max_num_locs_per_sample=bench.MAX_LOCS, device=dev)
    return S, d, m


def check_worker(out):
    """Loss and voxel gradients of each CHECKS case, to out.npz; the magnitude bound of atomic_f5 too."""
    import ctypes
    import numpy as np
    import torch
    from spsg_b200 import _native as N
    from spsg_b200 import losses as L
    from spsg_b200 import raycast_rgbd_cuda as rc
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {}
    for case in CHECKS:
        views = 1 if case == "det_f1" else F
        S, d, m = _inputs(dev, views)
        m.flags = N.SPSG_FLAG_DETERMINISTIC_GRADS if case.startswith("det") else 0
        cw = torch.tensor(S.CLASS_WEIGHTS, dtype=torch.float32, device=dev)
        targets = (d["t_depth"], d["t_color"], None, d["t_label"], cw, S.VOXELSIZE, (1.0, 1.0, 1.0))
        ups = None
        if case.endswith("upstream"):
            g = torch.Generator(device=dev).manual_seed(3)
            shape = (B * views, S.HEIGHT, S.WIDTH)
            ups = (torch.randn(shape + (3,), device=dev, generator=g) * 1e-6, None, None,
                   torch.randn(shape + (14,), device=dev, generator=g) * 1e-6)
        n = d["locs"].shape[0]
        p, tg, loss_out = L.fused_forward(m, d["locs"], d["sdf"], d["color"], d["normal"], d["semantic"], d["view"],
                                          d["intr"], targets, True)
        L.fused_backward(m, p, tg, loss_out, torch.ones((), device=dev), True, upstream=ups)
        for name, t in zip(("d_sdf", "d_color", "d_normal", "d_semantic"), L._voxel_grads(m, p, n)):
            res[case + "/" + name] = t.cpu().numpy()
        res[case + "/loss_out"] = loss_out.cpu().numpy()
        if case == "atomic_f5":
            # sum_f |mean_f| <= sum_f mean_f |g|: the plain deterministic gather of the absolute per-pixel gradients
            I = B * views
            imgs = [x[:I] for x in (m.image_color, m.image_depth, m.image_normal, m.image_semantic)]
            g_col, g_dep, g_sem = (torch.empty_like(x) for x in (imgs[0], imgs[1], imgs[3]))
            N.check(N.lib.spsg_losses2d_backward(ctypes.byref(tg), N.ptr(imgs[0]), N.ptr(imgs[1]), N.ptr(imgs[3]),
                                                 imgs[1].numel(), N.ptr(loss_out), N.ptr(torch.ones((), device=dev)),
                                                 N.ptr(g_col), N.ptr(g_dep), N.ptr(g_sem), rc._stream(dev)))
            dims = m.dims3d
            rc.backward(g_col.abs(), g_dep.abs(), torch.zeros_like(imgs[2]), g_sem.abs(), m.sparse_mapping,
                        m.mapping3dto2d, m.mapping3dto2d_num, [B, dims[2], dims[1], dims[0], n], m.d_color, m.d_depth,
                        m.d_normal, m.d_semantic, views_per_chunk=views, grads_cleared=False,
                        workspace_owner=m.workspace, flags=m.flags)
            for name, t in zip(("d_sdf", "d_color", "d_normal", "d_semantic"), L._voxel_grads(m, p, n)):
                res[case + "/mag_" + name] = t.cpu().numpy()
        del m
        torch.cuda.empty_cache()
    np.savez(out, **res)


def time_worker(out, min_window_s):
    """One window of each: fused-gather kernel time (timing hook, eager steps) and graph-replayed step time."""
    import time
    import torch
    import bench
    from spsg_b200 import _native as N
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    num_sets, _ = bench.auto_sets(B, F)
    o = bench.Ours(dev, 0, B, F, num_sets)
    for i in range(10):
        o.step_fused(i)
    torch.cuda.synchronize()
    N.timing_read(1)
    N.timing_enable(True)
    t0, i = time.perf_counter(), 0
    while time.perf_counter() - t0 < min_window_s or i < 50:
        o.step_fused(i)
        i += 1
        if i % 50 == 0:
            torch.cuda.synchronize()
    torch.cuda.synchronize()
    N.timing_enable(False)
    ms, launches = N.timing_read(1)
    graph = bench.capture_rotation(o.step_fused, num_sets, dev, 3)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    graph.replay()
    b.record()
    torch.cuda.synchronize()
    reps = max(2, int(min_window_s * 1000.0 / max(a.elapsed_time(b), 1e-3)) + 1)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        graph.replay()
    b.record()
    torch.cuda.synchronize()
    res = {"gather_us": ms / launches * 1e3, "gather_launches": launches,
           "step_ms": a.elapsed_time(b) / (reps * num_sets), "steps": reps * num_sets, "input_sets": num_sets}
    with open(out, "w") as f:
        json.dump(res, f)


# ---------------------------------------------------------------------------------------------------------------------
# driver
# ---------------------------------------------------------------------------------------------------------------------

def run_worker(lib, args):
    env = dict(os.environ, SPSG_RAYCAST_LIB=lib)
    subprocess.run([sys.executable, os.path.abspath(__file__)] + args, env=env, check=True, cwd=ROOT)


def device_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # no nvidia-smi on the PATH
        q = "unknown (%s)" % type(e).__name__
    return {"device": name, "power_limit, max_sm_clock": q}


def ulp_diff(a, b):
    """|a - b| in fp32 ulps (same-sign ordering of the bit patterns); NaN pairs count as equal."""
    import numpy as np
    ia, ib = a.view(np.int32).astype(np.int64), b.view(np.int32).astype(np.int64)
    ia = np.where(ia < 0, -(ia & 0x7fffffff), ia)
    ib = np.where(ib < 0, -(ib & 0x7fffffff), ib)
    d = np.abs(ia - ib)
    return np.where(np.isnan(a) & np.isnan(b), 0, d)


def compare(pa, pb):
    import numpy as np
    P, C = np.load(pa), np.load(pb)
    out, ok = {}, True
    for case in CHECKS:
        r = {}
        for name in ("loss_out", "d_sdf", "d_color", "d_normal", "d_semantic"):
            a, b = P[case + "/" + name], C[case + "/" + name]
            if case == "atomic_f5" and name != "loss_out":
                mag = P[case + "/mag_" + name].astype(np.float64)
                bound = 2 * (F - 1) * 2.0 ** -24 * mag + 2.0 ** -126
                err = np.abs(a.astype(np.float64) - b.astype(np.float64))
                outside = int((~(err <= bound) & ~(np.isnan(a) & np.isnan(b))).sum())
                r[name] = {"outside_bound": outside, "max_err_over_bound": float(np.nanmax(err / bound)) if a.size else 0.0}
                ok = ok and outside == 0
            else:
                u = ulp_diff(a, b)
                r[name] = {"entries": int(a.size), "differing": int((u != 0).sum()), "ties_1ulp": int((u == 1).sum()),
                           "beyond_1ulp": int((u > 1).sum())}
                ok = ok and (r[name]["beyond_1ulp"] == 0 if name != "loss_out" else r[name]["differing"] == 0)
        out[case] = r
    return out, ok


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--build-parent", metavar="REV", help="compile REV's native sources to build/ab_parent/ and exit")
    ap.add_argument("--out", default=None, help="directory for gather_ab.json")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--min-window-s", type=float, default=0.5)
    ap.add_argument("--worker", choices=["check", "time"], help=argparse.SUPPRESS)
    ap.add_argument("--worker-out", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.build_parent:
        build_parent(args.build_parent)
        return 0
    if args.worker == "check":
        check_worker(args.worker_out)
        return 0
    if args.worker == "time":
        time_worker(args.worker_out, args.min_window_s)
        return 0
    for lib in (PARENT_LIB, CURRENT_LIB):
        if not os.path.isfile(lib):
            sys.exit("missing %s (build it first: --build-parent REV, or __graft_entry__.build())" % lib)
    rev = os.path.join(os.path.dirname(PARENT_LIB), "REVISION")
    result = dict(device_info(), workload="c3", chunks=B, views=F,
                  parent=open(rev).read().strip() if os.path.isfile(rev) else "unknown")
    arms = {"parent": PARENT_LIB, "current": CURRENT_LIB}
    tmp = tempfile.mkdtemp()
    try:
        for arm, lib in arms.items():
            run_worker(lib, ["--worker", "check", "--worker-out", os.path.join(tmp, arm + ".npz")])
        result["checks"], ok = compare(os.path.join(tmp, "parent.npz"), os.path.join(tmp, "current.npz"))
        windows = {arm: [] for arm in arms}
        for r in range(args.rounds):
            for arm, lib in (list(arms.items()) if r % 2 == 0 else list(arms.items())[::-1]):
                path = os.path.join(tmp, "%s_%d.json" % (arm, r))
                run_worker(lib, ["--worker", "time", "--worker-out", path, "--min-window-s", str(args.min_window_s)])
                with open(path) as f:
                    windows[arm].append(json.load(f))
    finally:
        shutil.rmtree(tmp)
    result["windows"] = windows
    for key in ("gather_us", "step_ms"):
        result[key] = {arm: statistics.median(w[key] for w in windows[arm]) for arm in arms}
        result[key + "_spread"] = {arm: max(w[key] for w in windows[arm]) - min(w[key] for w in windows[arm])
                                   for arm in arms}
    result["gather_us_saved"] = result["gather_us"]["parent"] - result["gather_us"]["current"]
    result["step_speedup"] = result["step_ms"]["parent"] / result["step_ms"]["current"]
    result["checks_ok"] = ok
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "gather_ab.json"), "w") as f:
            f.write(line + "\n")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
