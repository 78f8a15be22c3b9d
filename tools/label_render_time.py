#!/usr/bin/env python
"""Label render (RaycastRGBD.render_labels, spsg_raycast_labels) against the route it replaces, on one GPU.

  target   the training step's target labels at C3 (8 chunks x 5 views, 320x256, bench.py's seeded chunks and cameras) for
           C = 14, 41, 64, from the target's sparse rows (locs, SDF) and one uint8 label per voxel:
             old  shared normals (compute_normals_sparse), the (N, C) float one-hot, the full raycast (colour, depth,
                  normal and C-channel images, voxel -> pixel registration, work list), labels_from_render
             new  render_labels
           (the sparsification of the target SDF and the gather of its labels, common to both, are outside the window;
           so is the old route's colour gather)
  room     one whole room of bench.py --workload c5 (128x256x320, 64x64 windows, stride 32, 5 views 320x256, 8 windows
           per launch), render_room against the previous render_room (normals + full render + labels_from_render of the
           semantic image), restated in tests/test_gpu_label_render.old_render_room.

Both routes run eagerly, as their callers launch them.  Old and new alternate within every round; each arm's time is the
median over rounds of CUDA-event windows of >= --min-window-s.  Outputs are compared (labels and histograms, bit for
bit) before timing.  Records the device name and power limit (read only).

    python tools/label_render_time.py [--out DIR] [--rounds 5] [--min-window-s 0.5]
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn.functional as Fn  # noqa: E402

from tools.upstream_time import B, F, power_limit  # noqa: E402

CLASSES = (14, 41, 64)


class Target:
    def __init__(self, dev, num_sets, C):
        import bench
        from spsg_b200 import synthetic as S
        from spsg_b200.raycast_rgbd import RaycastRGBD
        self.S, self.C = S, C
        self.sets = [{k: v.to(dev) for k, v in h.items()} for h in bench.make_host_sets(num_sets, B, F, 0)]
        g = torch.Generator(device=dev).manual_seed(C)
        for d in self.sets:
            d["labels"] = torch.randint(0, C + 1, (d["locs"].shape[0],), device=dev, generator=g).to(torch.uint8)
        self.mods = [RaycastRGBD(B, S.DIMS_ZYX, S.WIDTH, S.HEIGHT, S.DEPTH_MIN, S.DEPTH_MAX, S.THRESH_SAMPLE_DIST,
                                 S.RAY_INCREMENT, max_num_frames=F, max_num_locs_per_sample=bench.MAX_LOCS, device=dev,
                                 num_classes=C) for _ in self.sets]

    def old(self, i):
        from spsg_b200 import losses, normals
        k = i % len(self.sets)
        d, m = self.sets[k], self.mods[k]
        nrm = normals.compute_normals_sparse(d["locs"], d["sdf"], self.S.DIMS_ZYX, num_chunks=B)
        onehot = Fn.one_hot(d["labels"].long(), self.C + 1)[..., :-1].float().contiguous()
        _, _, _, sem = m(d["locs"], d["sdf"], d["color"], nrm, onehot, d["view"], d["intr"])
        return losses.labels_from_render(sem)

    def new(self, i):
        k = i % len(self.sets)
        d, m = self.sets[k], self.mods[k]
        return m.render_labels(d["locs"], d["sdf"], d["labels"], d["view"], d["intr"])


def timed(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for r in range(reps):
        fn(r)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def alternate(arms, rounds, min_s):
    reps = {}
    for name, fn in arms.items():
        for r in range(3):
            fn(r)  # warm-up: modules, workspaces, the caching allocator
        one = timed(fn, 2)
        reps[name] = max(2, int(min_s * 1000.0 / max(one, 1e-3)) + 1)
    ms = {name: [] for name in arms}
    for _ in range(rounds):
        for name, fn in arms.items():
            ms[name].append(timed(fn, reps[name]))
    return {name: statistics.median(t) for name, t in ms.items()}, ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="directory for label_render_time.json")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--min-window-s", type=float, default=0.5)
    args = ap.parse_args()
    import bench
    from spsg_b200 import room as R
    from tests.test_gpu_label_render import old_render_room
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    num_sets, _ = bench.auto_sets(B, F)
    result = {"device": torch.cuda.get_device_name(dev), "power_limit": power_limit(), "chunks": B, "views": F,
              "input_sets": num_sets, "target": {}}
    for C in CLASSES:
        t = Target(dev, num_sets, C)
        for i in range(num_sets):
            a, b = t.old(i).clone(), t.new(i)
            assert torch.equal(a, b), "C=%d set %d: label maps differ" % (C, i)
        med, windows = alternate({"old": t.old, "new": t.new}, args.rounds, args.min_window_s)
        result["target"]["c%d" % C] = {"ms": med, "ms_rounds": windows, "speedup": med["old"] / med["new"]}
        del t
        torch.cuda.empty_cache()

    dims = (128, 256, 320)
    room = R.synthetic_room_sdf(dims, dev)
    predict = R.synthetic_predictor(room)
    windows_ = R.chunk_windows(dims)
    predict.prepare_groups([windows_[s:s + 8] for s in range(0, len(windows_), 8)], (64, 64))
    kw = dict(views_per_chunk=5, chunks_per_launch=8)
    new_out = R.render_room(predict, dims, dev, keep_images=True, **kw)
    old_hist, old_images = old_render_room(predict, dims, dev, **kw)
    assert (new_out["label_hist"] == old_hist).all(), "room histograms differ"
    assert all(torch.equal(a, b) for (_, a), (_, b) in zip(new_out["images"], old_images)), "room label maps differ"
    arms = {"old": lambda r: old_render_room(predict, dims, dev, keep_images=False, **kw),
            "new": lambda r: R.render_room(predict, dims, dev, **kw)}
    med, rounds = alternate(arms, args.rounds, args.min_window_s)
    result["room"] = {"ms": med, "ms_rounds": rounds, "speedup": med["old"] / med["new"], "rays": new_out["rays"],
                      "label_hist": new_out["label_hist"].tolist()}
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "label_render_time.json"), "w") as f:
            f.write(line + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
