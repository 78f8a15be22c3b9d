#!/usr/bin/env python
"""Cost of the all-pixels mode (SPSG_FLAG_ALL_PIXELS) on the fused forward + backward (spsg_raycast_forward_loss,
spsg_raycast_backward_loss; all three 2D loss terms on) at C3 (8 chunks x 5 views, 320x256), four arms per camera set:

  default     the 64-entry voxel -> pixel table, sums in double in any order
  det         the same with SPSG_FLAG_DETERMINISTIC (canonical tables, overflowed rows rebuilt from the hit records)
  all         SPSG_FLAG_ALL_PIXELS: no table, every pixel of a row gathered from segments built in the backward
  all_det     SPSG_FLAG_ALL_PIXELS | SPSG_FLAG_DETERMINISTIC (segments sorted ascending)

on bench.py's seeded cameras (c3_*, 1.5 m from every surface: no row reaches 64 pixels) and on cameras 15-25 voxels
(0.3-0.5 m) in front of a wall (close_*, most rows over 64 pixels).  Timing as tools/deterministic_time.py: one step per
input set, captured into a CUDA graph, rotated over >= 2 input sets, CUDA-event windows of >= 0.5 s, arms alternated in one
process, median of three windows.  Records the device name and power limit (read only) and, per camera set, the rows that
received pixels, the rows over 64 and the largest row.

    python tools/all_pixels_time.py [--out DIR] [--windows 3] [--min-window-s 0.5]
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from tools.deterministic_time import close_views  # noqa: E402
from tools.upstream_time import B, F, capture, power_limit, window  # noqa: E402

ARMS = ("default", "det", "all", "all_det")


class Arms:
    def __init__(self, dev, num_sets):
        import bench
        from spsg_b200 import _native as N
        from spsg_b200 import synthetic as S
        from spsg_b200.raycast_rgbd import RaycastRGBD
        self.S, self.N, self.dev = S, N, dev
        self.sets, self.mods = [], {}
        for k, h in enumerate(bench.make_host_sets(num_sets, B, F, 0)):
            d = {key: v.to(dev) for key, v in h.items()}
            d["view_close"] = torch.from_numpy(close_views(B * F, 100 + k)).to(dev)
            self.sets.append(d)
        for arm in ARMS:
            table = not arm.startswith("all")
            self.mods[arm] = [RaycastRGBD(B, S.DIMS_ZYX, S.WIDTH, S.HEIGHT, S.DEPTH_MIN, S.DEPTH_MAX, S.THRESH_SAMPLE_DIST,
                                          S.RAY_INCREMENT, max_num_frames=F, max_num_locs_per_sample=bench.MAX_LOCS,
                                          max_pixels_per_voxel=64 if table else None, device=dev) for _ in self.sets]
            for m in self.mods[arm]:
                m.flags |= N.SPSG_FLAG_DETERMINISTIC if arm.endswith("det") else 0
        self.cw = torch.tensor(S.CLASS_WEIGHTS, dtype=torch.float32, device=dev)
        self.one = torch.ones((), device=dev)

    def step(self, i, view, arm):
        from spsg_b200 import losses as L
        k = i % len(self.sets)
        d, m = self.sets[k], self.mods[arm][k]
        targets = (d["t_depth"], d["t_color"], None, d["t_label"], self.cw, self.S.VOXELSIZE, (1.0, 1.0, 1.0))
        p, tg, loss_out = L.fused_forward(m, d["locs"], d["sdf"], d["color"], d["normal"], d["semantic"], d[view],
                                          d["intr"], targets, True)
        L.fused_backward(m, p, tg, loss_out, self.one, True)

    def rows(self, view):
        """(rows that received pixels, rows over 64, largest row) of set 0"""
        self.step(0, view, "all")
        torch.cuda.synchronize()
        m, n = self.mods["all"][0], self.sets[0]["locs"].shape[0]
        num = m.mapping3dto2d_num[:F * n]
        return int((num > 0).sum()), int((num > 64).sum()), int(num.max())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="directory for all_pixels_time.json")
    ap.add_argument("--windows", type=int, default=3)
    ap.add_argument("--min-window-s", type=float, default=0.5)
    args = ap.parse_args()
    import bench
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    num_sets, per_set_mb = bench.auto_sets(B, F)
    v = Arms(dev, num_sets)
    result = {"device": torch.cuda.get_device_name(dev), "power_limit": power_limit(), "chunks": B, "views": F,
              "width": v.S.WIDTH, "height": v.S.HEIGHT, "input_sets": num_sets, "input_set_mb": per_set_mb,
              "rows": {"c3": v.rows("view"), "close": v.rows("view_close")}}
    names = {}
    for cams, view in (("c3", "view"), ("close", "view_close")):
        for arm in ARMS:
            names["%s_%s" % (cams, arm)] = (lambda view, arm: lambda i: v.step(i, view, arm))(view, arm)
    graphs, reps = {}, {}
    for name, step in names.items():
        graphs[name], mode = capture(step, num_sets, dev)
        result.setdefault("replay", {})[name] = mode
        one = window(graphs[name], step, num_sets, 2) / 2
        reps[name] = max(2, int(args.min_window_s * 1000.0 / max(one, 1e-3)) + 1)
    ms = {name: [] for name in names}
    for _ in range(args.windows):
        for name, step in names.items():
            ms[name].append(window(graphs[name], step, num_sets, reps[name]) / (reps[name] * num_sets))
    result["step_ms"] = {name: statistics.median(t) for name, t in ms.items()}
    result["step_ms_windows"] = ms
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "all_pixels_time.json"), "w") as f:
            f.write(line + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
