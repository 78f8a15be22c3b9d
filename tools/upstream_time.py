#!/usr/bin/env python
"""Cost of an image-space term (GAN / style) on the prediction render at C3 (8 chunks x 5 views, 320x256; bench.py's seeded
synthetic inputs, all three 2D loss terms on, seeded colour and normal upstream gradient images):

  (a) fused + upstream   spsg_raycast_forward_loss, then spsg_raycast_backward_loss_upstream (the colour and normal
                         gradient images gathered in the same launch as the recomputed loss gradients)
  (b) un-fused           raycast forward, losses_2d forward + backward (gradient images), the upstream images added,
                         plain raycast backward
  (c) fused, no upstream the existing pair (bench.py's headline step), for reference

Each variant is one step per input set, captured into a CUDA graph (eager replay if capture is refused) and rotated over
>= 2 input sets so that the working set exceeds the 126 MB L2.  CUDA-event windows of >= 0.5 s, the variants alternated
in one process, median of three windows each.  Also checks that (a) and (b) give the same loss and voxel gradients
(1e-3) at the timed size, and records the device name and power limit (read only).

    python tools/upstream_time.py [--out DIR] [--windows 3] [--min-window-s 0.5]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

B, F = 8, 5


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        return out.stdout.strip() or None
    except Exception as e:  # no nvidia-smi on the PATH
        return "unknown (%s)" % type(e).__name__


class Variants:
    def __init__(self, dev, num_sets):
        import bench
        from spsg_b200 import synthetic as S
        from spsg_b200.raycast_rgbd import RaycastRGBD
        self.S, self.dev = S, dev
        self.sets, self.mods, self.up = [], [], []
        for k, h in enumerate(bench.make_host_sets(num_sets, B, F, 0)):
            self.sets.append({key: v.to(dev) for key, v in h.items()})
            self.mods.append(RaycastRGBD(B, S.DIMS_ZYX, S.WIDTH, S.HEIGHT, S.DEPTH_MIN, S.DEPTH_MAX, S.THRESH_SAMPLE_DIST,
                                         S.RAY_INCREMENT, max_num_frames=F, max_num_locs_per_sample=bench.MAX_LOCS,
                                         device=dev))
            g = torch.Generator(device=dev).manual_seed(100 + k)
            shape = (B * F, S.HEIGHT, S.WIDTH, 3)
            self.up.append((torch.randn(shape, device=dev, generator=g) * 1e-6,
                            torch.randn(shape, device=dev, generator=g) * 1e-6))
        self.cw = torch.tensor(S.CLASS_WEIGHTS, dtype=torch.float32, device=dev)
        self.one = torch.ones((), device=dev)
        self.out = {}

    def _targets(self, d):
        return (d["t_depth"], d["t_color"], None, d["t_label"], self.cw, self.S.VOXELSIZE, (1.0, 1.0, 1.0))

    def fused(self, i, upstream=True):
        from spsg_b200 import losses as L
        k = i % len(self.sets)
        d, m = self.sets[k], self.mods[k]
        p, tg, loss_out = L.fused_forward(m, d["locs"], d["sdf"], d["color"], d["normal"], d["semantic"], d["view"],
                                          d["intr"], self._targets(d), True)
        up = (self.up[k][0], None, self.up[k][1], None) if upstream else None
        L.fused_backward(m, p, tg, loss_out, self.one, True, upstream=up)
        self.out[k] = loss_out[3]

    def plain_fused(self, i):
        self.fused(i, upstream=False)

    def unfused(self, i):
        from spsg_b200 import losses as L
        from spsg_b200 import raycast_rgbd_cuda as rcc
        S = self.S
        k = i % len(self.sets)
        d, m = self.sets[k], self.mods[k]
        n, I = d["locs"].shape[0], B * F
        opts = [S.WIDTH, S.HEIGHT, S.DEPTH_MIN, S.DEPTH_MAX, S.THRESH_SAMPLE_DIST, S.RAY_INCREMENT, S.DIMS_ZYX[2],
                S.DIMS_ZYX[1], S.DIMS_ZYX[0]]
        rcc.forward(m.sparse_mapping, d["locs"], d["sdf"], d["color"], d["normal"], d["semantic"], d["view"],
                    m.image_color, m.image_depth, m.image_normal, m.image_semantic, m.mapping3dto2d, m.mapping3dto2d_num,
                    d["intr"], opts, views_per_chunk=F, build_index=True,
                    clear_grads=(m.d_color, m.d_depth, m.d_normal, m.d_semantic), workspace_owner=m.workspace)
        col, dep, sem = (x[:I].detach().requires_grad_(True) for x in (m.image_color, m.image_depth, m.image_semantic))
        total, _ = L.losses_2d(col, dep, sem, images_depth=d["t_depth"], images_color=d["t_color"],
                               target2d_label=d["t_label"], weight_semantic_class=self.cw, voxelsize=S.VOXELSIZE)
        g_col, g_dep, g_sem = torch.autograd.grad(total, (col, dep, sem))
        rcc.backward(g_col + self.up[k][0], g_dep, self.up[k][1], g_sem, m.sparse_mapping, m.mapping3dto2d,
                     m.mapping3dto2d_num, [B, S.DIMS_ZYX[2], S.DIMS_ZYX[1], S.DIMS_ZYX[0], n], m.d_color, m.d_depth,
                     m.d_normal, m.d_semantic, views_per_chunk=F, grads_cleared=True, workspace_owner=m.workspace)
        self.out[k] = total.detach()

    def grads(self, k):
        n = self.sets[k]["locs"].shape[0]
        m = self.mods[k]
        return [t[:n].clone() for t in (m.d_depth, m.d_color, m.d_normal, m.d_semantic)]


def check_a_vs_b(v):
    v.fused(0)
    loss_a, ga = float(v.out[0]), v.grads(0)
    v.unfused(0)
    loss_b, gb = float(v.out[0]), v.grads(0)
    res = {"loss_a": loss_a, "loss_b": loss_b, "loss_rel": abs(loss_a - loss_b) / max(abs(loss_b), 1e-30)}
    ok = res["loss_rel"] <= 1e-5
    for name, a, b in zip(("sdf", "color", "normal", "semantic"), ga, gb):
        scale = float(b.abs().max())
        err = (a - b).abs()
        bad = int((err > 1e-3 * b.abs() + 1e-6 * scale).sum())
        res[name] = {"max_abs_err": float(err.max()), "scale": scale, "elements_outside_1e-3": bad}
        ok = ok and bad == 0 and scale > 0
    res["ok"] = ok
    return res


def capture(step, num_sets, dev):
    import bench
    try:
        return bench.capture_rotation(step, num_sets, dev, 3), "graph"
    except Exception as e:  # capture refused: replay eagerly
        torch.cuda.synchronize()
        return None, "eager (%s)" % type(e).__name__


def window(graph, step, num_sets, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for r in range(reps):
        if graph is not None:
            graph.replay()
        else:
            for i in range(num_sets):
                step(i)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="directory for upstream_time.json")
    ap.add_argument("--windows", type=int, default=3)
    ap.add_argument("--min-window-s", type=float, default=0.5)
    args = ap.parse_args()
    import bench
    from spsg_b200 import _native  # noqa: F401  (fails loudly without the library)
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    num_sets, per_set_mb = bench.auto_sets(B, F)
    v = Variants(dev, num_sets)
    result = {"device": torch.cuda.get_device_name(dev), "power_limit": power_limit(), "workload": "c3",
              "chunks": B, "views": F, "width": v.S.WIDTH, "height": v.S.HEIGHT, "input_sets": num_sets,
              "input_set_mb": per_set_mb, "check_a_vs_b": check_a_vs_b(v)}
    names = {"a_fused_upstream": v.fused, "b_unfused": v.unfused, "c_fused_no_upstream": v.plain_fused}
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
    result["steps_per_window"] = {name: reps[name] * num_sets for name in names}
    result["a_over_b"] = result["step_ms"]["a_fused_upstream"] / result["step_ms"]["b_unfused"]
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "upstream_time.json"), "w") as f:
            f.write(line + "\n")
    return 0 if result["check_a_vs_b"]["ok"] else 1


if __name__ == "__main__":
    sys.exit(main())
