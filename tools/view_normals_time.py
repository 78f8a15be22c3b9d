#!/usr/bin/env python
"""Cost of per-view normals (SPSG_FLAG_VIEW_NORMALS) at C3 (8 chunks x 5 views, 320x256; bench.py's seeded synthetic
inputs, all three 2D loss terms on):

  raycast_shared   fused forward + backward (spsg_raycast_forward_loss, spsg_raycast_backward_loss) with (N,3) normals
  raycast_views    the same with (N,5,3) normals: the per-view forward and gather instantiations, N*F normal rows
  normals_f1       the normals op, forward + backward (spsg_normals_forward / _backward), one rotation per chunk
  normals_f5       spsg_normals_forward_views / _backward_views with F = 5, one rotation per image

Each arm is one step per input set, captured into a CUDA graph (eager replay if capture is refused) and rotated over >= 2
input sets so that the working set exceeds the 126 MB L2.  CUDA-event windows of >= 0.5 s, the arms alternated in one
process, median of three windows each.  Records the device name and power limit (read only).

    python tools/view_normals_time.py [--out DIR] [--windows 3] [--min-window-s 0.5]
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


class Arms:
    def __init__(self, dev, num_sets):
        import bench
        from spsg_b200 import synthetic as S
        from spsg_b200.raycast_rgbd import RaycastRGBD
        self.S, self.dev = S, dev
        self.sets, self.mods, self.scratch = [], [], []
        for h in bench.make_host_sets(num_sets, B, F, 0):
            d = {key: v.to(dev) for key, v in h.items()}
            n = d["locs"].shape[0]
            # a distinct row per view (the values do not change the work)
            d["normal_views"] = torch.stack([d["normal"].roll(f, 1) for f in range(F)], 1).contiguous()
            d["transform"] = torch.inverse(d["view"]).contiguous()
            d["transform1"] = d["transform"][::F].contiguous()
            self.sets.append(d)
            self.mods.append(RaycastRGBD(B, S.DIMS_ZYX, S.WIDTH, S.HEIGHT, S.DEPTH_MIN, S.DEPTH_MAX, S.THRESH_SAMPLE_DIST,
                                         S.RAY_INCREMENT, max_num_frames=F, max_num_locs_per_sample=bench.MAX_LOCS,
                                         device=dev))
            g = torch.Generator(device=dev).manual_seed(7)
            self.scratch.append(dict(
                index=torch.empty((B,) + tuple(S.DIMS_ZYX), dtype=torch.int32, device=dev),
                out1=torch.empty(n, 3, device=dev), out5=torch.empty(n, F, 3, device=dev),
                g1=torch.randn(n, 3, device=dev, generator=g), g5=torch.randn(n, F, 3, device=dev, generator=g),
                u=torch.empty(n, 3, device=dev), d_sdf=torch.empty(n, 1, device=dev)))
        self.cw = torch.tensor(S.CLASS_WEIGHTS, dtype=torch.float32, device=dev)
        self.one = torch.ones((), device=dev)

    def _raycast(self, i, normals):
        from spsg_b200 import losses as L
        k = i % len(self.sets)
        d, m = self.sets[k], self.mods[k]
        targets = (d["t_depth"], d["t_color"], None, d["t_label"], self.cw, self.S.VOXELSIZE, (1.0, 1.0, 1.0))
        p, tg, loss_out = L.fused_forward(m, d["locs"], d["sdf"], d["color"], d[normals], d["semantic"], d["view"],
                                          d["intr"], targets, True)
        L.fused_backward(m, p, tg, loss_out, self.one, True)

    def raycast_shared(self, i):
        self._raycast(i, "normal")

    def raycast_views(self, i):
        self._raycast(i, "normal_views")

    def _normals(self, i, views):
        from spsg_b200 import _native as N
        k = i % len(self.sets)
        d, s = self.sets[k], self.scratch[k]
        n, dims = d["locs"].shape[0], self.S.DIMS_ZYX
        st = torch.cuda.current_stream(self.dev).cuda_stream
        ptr = N.ptr
        if views == 1:
            N.check(N.lib.spsg_normals_forward(ptr(d["locs"]), n, ptr(d["sdf"]), ptr(d["transform1"]), ptr(s["index"]),
                                               B, dims[0], dims[1], dims[2], ptr(s["out1"]), st))
            N.check(N.lib.spsg_normals_backward(ptr(d["locs"]), n, ptr(d["sdf"]), ptr(d["transform1"]), ptr(s["index"]),
                                                B, dims[0], dims[1], dims[2], ptr(s["g1"]), ptr(s["u"]), ptr(s["d_sdf"]),
                                                st))
        else:
            N.check(N.lib.spsg_normals_forward_views(ptr(d["locs"]), n, ptr(d["sdf"]), ptr(d["transform"]), F,
                                                     ptr(s["index"]), B, dims[0], dims[1], dims[2], ptr(s["out5"]), st))
            N.check(N.lib.spsg_normals_backward_views(ptr(d["locs"]), n, ptr(d["sdf"]), ptr(d["transform"]), F,
                                                      ptr(s["index"]), B, dims[0], dims[1], dims[2], ptr(s["g5"]),
                                                      ptr(s["u"]), ptr(s["d_sdf"]), st))

    def normals_f1(self, i):
        self._normals(i, 1)

    def normals_f5(self, i):
        self._normals(i, F)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="directory for view_normals_time.json")
    ap.add_argument("--windows", type=int, default=3)
    ap.add_argument("--min-window-s", type=float, default=0.5)
    args = ap.parse_args()
    import bench
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    num_sets, per_set_mb = bench.auto_sets(B, F)
    v = Arms(dev, num_sets)
    result = {"device": torch.cuda.get_device_name(dev), "power_limit": power_limit(), "workload": "c3",
              "chunks": B, "views": F, "width": v.S.WIDTH, "height": v.S.HEIGHT, "input_sets": num_sets,
              "input_set_mb": per_set_mb}
    names = {"raycast_shared": v.raycast_shared, "raycast_views": v.raycast_views, "normals_f1": v.normals_f1,
             "normals_f5": v.normals_f5}
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
    result["views_over_shared"] = result["step_ms"]["raycast_views"] / result["step_ms"]["raycast_shared"]
    result["normals_f5_over_f1"] = result["step_ms"]["normals_f5"] / result["step_ms"]["normals_f1"]
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "view_normals_time.json"), "w") as f:
            f.write(line + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
