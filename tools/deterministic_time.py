#!/usr/bin/env python
"""Cost of deterministic mode (SPSG_FLAG_DETERMINISTIC) on the fused forward + backward (spsg_raycast_forward_loss,
spsg_raycast_backward_loss; all three 2D loss terms on) at C3 (8 chunks x 5 views, 320x256):

  c3_default / c3_det        bench.py's seeded synthetic inputs and cameras (1.5 m from every surface)
  close_default / close_det  the same chunks and targets, cameras 15-25 voxels (0.3-0.5 m) in front of a wall: most
                             (voxel, view) rows get more pixels than their 64-entry table, and are rebuilt from the hits

Each arm is one step per input set, captured into a CUDA graph (eager replay if capture is refused) and rotated over >= 2
input sets so that the working set exceeds the 126 MB L2.  CUDA-event windows of >= 0.5 s, the arms alternated in one
process, median of three windows each.  Records the device name and power limit (read only) and, per workload, how many
(voxel, view) rows received pixels and how many overflowed.

    python tools/deterministic_time.py [--out DIR] [--windows 3] [--min-window-s 0.5]
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from tools.upstream_time import B, F, capture, power_limit, window  # noqa: E402


def close_views(images, seed):
    """camera->grid matrices 15-25 voxels in front of the synthetic room's walls, above the sphere and the box"""
    from spsg_b200 import synthetic as S
    rng = np.random.default_rng(seed)
    mats = []
    for _ in range(images):
        d, a, z = rng.uniform(15.0, 25.0), rng.uniform(15.0, 45.0), rng.uniform(55.0, 75.0)
        if rng.random() < 0.5:
            mats.append(S.look_at((a, 56.7 - d, z), (a + rng.uniform(-6, 6), 62.0, z + rng.uniform(-8, 4))))
        else:
            mats.append(S.look_at((57.2 - d, a, z), (62.0, a + rng.uniform(-6, 6), z + rng.uniform(-8, 4))))
    return np.stack(mats).astype(np.float32)


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
        for det in (False, True):
            self.mods[det] = [RaycastRGBD(B, S.DIMS_ZYX, S.WIDTH, S.HEIGHT, S.DEPTH_MIN, S.DEPTH_MAX, S.THRESH_SAMPLE_DIST,
                                          S.RAY_INCREMENT, max_num_frames=F, max_num_locs_per_sample=bench.MAX_LOCS,
                                          device=dev) for _ in self.sets]
            for m in self.mods[det]:
                m.flags = N.SPSG_FLAG_DETERMINISTIC if det else 0
        self.cw = torch.tensor(S.CLASS_WEIGHTS, dtype=torch.float32, device=dev)
        self.one = torch.ones((), device=dev)

    def step(self, i, view, det):
        from spsg_b200 import losses as L
        k = i % len(self.sets)
        d, m = self.sets[k], self.mods[det][k]
        targets = (d["t_depth"], d["t_color"], None, d["t_label"], self.cw, self.S.VOXELSIZE, (1.0, 1.0, 1.0))
        p, tg, loss_out = L.fused_forward(m, d["locs"], d["sdf"], d["color"], d["normal"], d["semantic"], d[view],
                                          d["intr"], targets, True)
        L.fused_backward(m, p, tg, loss_out, self.one, True)

    def rows(self, view):
        """(rows that received pixels, rows over max_pixels_per_voxel) of set 0, from a deterministic step"""
        self.step(0, view, True)
        torch.cuda.synchronize()
        m, n = self.mods[True][0], self.sets[0]["locs"].shape[0]
        num = m.mapping3dto2d_num[:F * n]
        return int((num > 0).sum()), int((num > m.mapping3dto2d.shape[1]).sum())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="directory for deterministic_time.json")
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
    names = {"c3_default": lambda i: v.step(i, "view", False), "c3_det": lambda i: v.step(i, "view", True),
             "close_default": lambda i: v.step(i, "view_close", False),
             "close_det": lambda i: v.step(i, "view_close", True)}
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
    result["c3_det_over_default"] = result["step_ms"]["c3_det"] / result["step_ms"]["c3_default"]
    result["close_det_over_default"] = result["step_ms"]["close_det"] / result["step_ms"]["close_default"]
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "deterministic_time.json"), "w") as f:
            f.write(line + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
