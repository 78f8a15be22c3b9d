#!/usr/bin/env python
"""Eval render (losses.evaluate_2d, spsg_raycast_eval) against today's evaluation route, on one GPU.

At C3 (8 chunks x 5 views, 320x256, bench.py's seeded chunks and cameras) for C = 14, 41, 64, from the prediction's sparse
rows (locs, SDF, colour, C logits) and seeded targets (depth, colour, labels 0..C):
    old  the normals op, render_with_2d_losses under no_grad (fused forward: images, registration, work list),
         labels_from_render of the semantic image, and a torch bincount confusion matrix
    new  evaluate_2d with the confusion matrix (labels_from_render of the logits rows included)
Both routes run eagerly.  Old and new alternate within every round; each arm's time is the median over rounds of
CUDA-event windows of >= --min-window-s.  Outputs are compared first (normalisers bit for bit, terms within 1e-6, the
confusion matrix exactly).  Records the device name and power limit (read only).

    python tools/eval_render_time.py [--out DIR] [--rounds 5] [--min-window-s 0.5]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from tools.label_render_time import alternate  # noqa: E402
from tools.upstream_time import B, F, power_limit  # noqa: E402

CLASSES = (14, 41, 64)


class Eval:
    def __init__(self, dev, num_sets, C):
        import bench
        from spsg_b200 import synthetic as S
        from spsg_b200.raycast_rgbd import RaycastRGBD
        self.S, self.C = S, C
        self.sets = [{k: v.to(dev) for k, v in h.items()} for h in bench.make_host_sets(num_sets, B, F, 0)]
        g = torch.Generator(device=dev).manual_seed(C)
        images = B * F
        for d in self.sets:
            n = d["locs"].shape[0]
            d["logits"] = (torch.randn(n, C, device=dev, generator=g) * 2.0).contiguous()
            d["tdepth"] = torch.rand(images, S.HEIGHT, S.WIDTH, device=dev, generator=g) * 3.0
            d["tcolor"] = torch.rand(images, S.HEIGHT, S.WIDTH, 3, device=dev, generator=g)
            d["tlabel"] = torch.randint(0, C + 1, (images, S.HEIGHT, S.WIDTH), device=dev, generator=g).to(torch.uint8)
        self.cw = torch.rand(C, device=dev, generator=g) + 0.5
        self.mods = [RaycastRGBD(B, S.DIMS_ZYX, S.WIDTH, S.HEIGHT, S.DEPTH_MIN, S.DEPTH_MAX, S.THRESH_SAMPLE_DIST,
                                 S.RAY_INCREMENT, max_num_frames=F, max_num_locs_per_sample=bench.MAX_LOCS, device=dev,
                                 num_classes=C) for _ in self.sets]

    def old(self, i):
        from spsg_b200 import losses, normals
        k = i % len(self.sets)
        d, m, C = self.sets[k], self.mods[k], self.C
        with torch.no_grad():
            nrm = normals.compute_normals_sparse(d["locs"], d["sdf"], self.S.DIMS_ZYX, num_chunks=B)
            total, terms, imgs = losses.render_with_2d_losses(
                m, d["locs"], d["sdf"], d["color"], nrm, d["logits"], d["view"], d["intr"], images_depth=d["tdepth"],
                images_color=d["tcolor"], target2d_label=d["tlabel"], weight_semantic_class=self.cw)
            lab = losses.labels_from_render(imgs[3])
            conf = torch.bincount(d["tlabel"].long().clamp(max=C).flatten() * (C + 1) + lab.long().flatten(),
                                  minlength=(C + 1) ** 2).view(C + 1, C + 1)
        return total, terms, conf

    def new(self, i):
        from spsg_b200 import losses
        k = i % len(self.sets)
        d, m = self.sets[k], self.mods[k]
        total, terms, conf, _ = losses.evaluate_2d(
            m, d["locs"], d["sdf"], d["color"], d["logits"], d["view"], d["intr"], images_depth=d["tdepth"],
            images_color=d["tcolor"], target2d_label=d["tlabel"], weight_semantic_class=self.cw)
        return total, terms, conf


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="directory for eval_render_time.json")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--min-window-s", type=float, default=0.5)
    args = ap.parse_args()
    import bench
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    num_sets, _ = bench.auto_sets(B, F)
    result = {"device": torch.cuda.get_device_name(dev), "power_limit": power_limit(), "chunks": B, "views": F,
              "input_sets": num_sets, "eval": {}}
    for C in CLASSES:
        t = Eval(dev, num_sets, C)
        for i in range(num_sets):
            ot, oterms, oc = (x.clone() for x in t.old(i))
            nt, nterms, nc = t.new(i)
            a = torch.cat([nterms, nt[None]]).double()
            b = torch.cat([oterms, ot[None]]).double()
            assert bool(((a - b).abs() <= 1e-6 * b.abs()).all()), "C=%d set %d: terms %s vs %s" % (C, i, a.tolist(), b.tolist())
            assert torch.equal(nc, oc), "C=%d set %d: confusion matrices differ" % (C, i)
        med, windows = alternate({"old": t.old, "new": t.new}, args.rounds, args.min_window_s)
        result["eval"]["c%d" % C] = {"ms": med, "ms_rounds": windows, "speedup": med["old"] / med["new"]}
        del t
        torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "eval_render_time.json"), "w") as f:
            f.write(line + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
