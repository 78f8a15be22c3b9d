#!/usr/bin/env python
"""Cost of the semantic class count C on the fused forward + backward (spsg_raycast_forward_loss,
spsg_raycast_backward_loss; all three 2D loss terms on) at C3 (8 chunks x 5 views, 320x256, bench.py's seeded cameras),
five arms:

  c14         C = 14, the 14-channel kernels
  c14_generic C = 14 with SPSG_FLAG_GENERIC_SEMANTIC: the C-generic kernels at the same C
  c20, c41, c64  the C-generic kernels at C = 20 (ScanNet), 41 (NYU40 / mpcat40) and 64 (the largest C)

The C-channel arms render the same voxels with seeded N(0, 2) logits and the same labels (0..14, all valid classes for
C > 14); class weights are bench.py's 14 followed by ones.  Timing as tools/all_pixels_time.py: one step per input set,
captured into a CUDA graph, rotated over >= 2 input sets, CUDA-event windows of >= 0.5 s, arms alternated in one process,
median of three windows.  Records the device name and power limit (read only).

    python tools/semantic_classes_time.py [--out DIR] [--windows 3] [--min-window-s 0.5]
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from tools.upstream_time import B, F, capture, power_limit, window  # noqa: E402

ARMS = {"c14": (14, False), "c14_generic": (14, True), "c20": (20, False), "c41": (41, False), "c64": (64, False)}


class Arms:
    def __init__(self, dev, num_sets):
        import bench
        from spsg_b200 import _native as N
        from spsg_b200 import synthetic as S
        from spsg_b200.raycast_rgbd import RaycastRGBD
        self.S, self.dev = S, dev
        self.sets = [{key: v.to(dev) for key, v in h.items()} for h in bench.make_host_sets(num_sets, B, F, 0)]
        self.mods, self.sem, self.cw = {}, {}, {}
        for arm, (c, generic) in ARMS.items():
            self.mods[arm] = [RaycastRGBD(B, S.DIMS_ZYX, S.WIDTH, S.HEIGHT, S.DEPTH_MIN, S.DEPTH_MAX, S.THRESH_SAMPLE_DIST,
                                          S.RAY_INCREMENT, max_num_frames=F, max_num_locs_per_sample=bench.MAX_LOCS,
                                          device=dev, num_classes=c) for _ in self.sets]
            for m in self.mods[arm]:
                m.flags |= N.SPSG_FLAG_GENERIC_SEMANTIC if generic else 0
            g = torch.Generator(device=dev).manual_seed(c)
            self.sem[arm] = [d["semantic"] if c == 14 else
                             torch.randn(d["locs"].shape[0], c, device=dev, generator=g) * 2.0 for d in self.sets]
            w = list(S.CLASS_WEIGHTS) + [1.0] * max(0, c - 14)
            self.cw[arm] = torch.tensor(w[:c], dtype=torch.float32, device=dev)
        self.one = torch.ones((), device=dev)

    def step(self, i, arm):
        from spsg_b200 import losses as L
        k = i % len(self.sets)
        d, m = self.sets[k], self.mods[arm][k]
        targets = (d["t_depth"], d["t_color"], None, d["t_label"], self.cw[arm], self.S.VOXELSIZE, (1.0, 1.0, 1.0))
        p, tg, loss_out = L.fused_forward(m, d["locs"], d["sdf"], d["color"], d["normal"], self.sem[arm][k], d["view"],
                                          d["intr"], targets, True)
        L.fused_backward(m, p, tg, loss_out, self.one, True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="directory for semantic_classes_time.json")
    ap.add_argument("--windows", type=int, default=3)
    ap.add_argument("--min-window-s", type=float, default=0.5)
    args = ap.parse_args()
    import bench
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    num_sets, per_set_mb = bench.auto_sets(B, F)
    v = Arms(dev, num_sets)
    result = {"device": torch.cuda.get_device_name(dev), "power_limit": power_limit(), "chunks": B, "views": F,
              "width": v.S.WIDTH, "height": v.S.HEIGHT, "input_sets": num_sets, "input_set_mb": per_set_mb}
    names = {arm: (lambda arm: lambda i: v.step(i, arm))(arm) for arm in ARMS}
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
        with open(os.path.join(args.out, "semantic_classes_time.json"), "w") as f:
            f.write(line + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
