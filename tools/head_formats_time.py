#!/usr/bin/env python
"""Time the producer glue on the heads a generator in channels_last_3d (and under bfloat16 autocast) produces, and the
training step with and without ``autocast_bf16``.  One process; prints the card's name and power limit with the numbers.

1. Glue alone, forward + backward (count, rows, gathers of SDF + colour + 14-class heads, the scatter backward) at the
   train leg's sizes: 8 chunks of 128x64x64, about 1 M voxels, synthetic heads from a seed.  For fp32-NDHWC and bf16-NDHWC
   heads: the copy route (``.float().contiguous()`` + the float32 NCDHW glue) against the in-place route; fp32 NCDHW heads
   as the unchanged reference point.  Routes alternate within each round; the median over rounds is reported.
2. The training step, fp32-NDHWC against bf16-autocast-NDHWC, on the reference generator where ``baseline/_ref`` is
   installed, else on a seeded Conv3d + BatchNorm3d stand-in of the reference's width (nf 20), labelled as such.

    python tools/head_formats_time.py [--rounds 7] [--iters 20] [--steps 8] [--json out.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn.functional as Fn  # noqa: E402

B, DIMS, T = 8, (128, 64, 64), 3.0


def card():
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.check_output(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                                        text=True).strip()
    except (OSError, subprocess.CalledProcessError):
        limit = "unknown"
    return name, limit


def glue_heads(dev, dtype, layout):
    """SDF (about a quarter of the cells within the truncation: ~1 M voxels), colour (3), semantics (14)"""
    g = torch.Generator(device=dev).manual_seed(11)
    sdf = (torch.rand(B, 1, *DIMS, generator=g, device=dev) * 2 - 1) * 12.0
    col = torch.rand(B, 3, *DIMS, generator=g, device=dev) * 2 - 1
    sem = torch.randn(B, 14, *DIMS, generator=g, device=dev)
    fmt = torch.channels_last_3d if layout == "ndhwc" else torch.contiguous_format
    return [t.to(dtype).contiguous(memory_format=fmt).requires_grad_(True) for t in (sdf, col, sem)]


def glue_once(heads, copy, grads):
    from spsg_b200 import sparsify
    ins = [h.float().contiguous() for h in heads] if copy else heads
    locs, *vals = sparsify.sparsify_predictions(ins[0], T, None, ins[1], ins[2])
    n = locs.shape[0]
    torch.autograd.backward(vals, [g[:n] for g in grads])
    return n


def time_glue(dev, rounds, iters):
    routes = {
        "fp32_ncdhw (original glue)": (torch.float32, "ncdhw", False),
        "fp32_ndhwc copy (.float().contiguous())": (torch.float32, "ndhwc", True),
        "fp32_ndhwc in place": (torch.float32, "ndhwc", False),
        "bf16_ndhwc copy (.float().contiguous())": (torch.bfloat16, "ndhwc", True),
        "bf16_ndhwc in place": (torch.bfloat16, "ndhwc", False),
    }
    heads = {k: glue_heads(dev, dt, lay) for k, (dt, lay, _) in routes.items()}
    cells = B * DIMS[0] * DIMS[1] * DIMS[2]
    g = torch.Generator(device=dev).manual_seed(3)
    grads = [torch.randn(cells // 2, c, generator=g, device=dev) for c in (1, 3, 14)]
    n = {}
    for k, (_, _, copy) in routes.items():   # warm-up: every shape the timed window uses
        for _ in range(3):
            n[k] = glue_once(heads[k], copy, grads)
    assert n[k] <= cells // 2
    ms = {k: [] for k in routes}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for _ in range(rounds):
        for k, (_, _, copy) in routes.items():
            torch.cuda.synchronize()
            ev[0].record()
            for _ in range(iters):
                for h in heads[k]:
                    h.grad = None
                glue_once(heads[k], copy, grads)
            ev[1].record()
            torch.cuda.synchronize()
            ms[k].append(ev[0].elapsed_time(ev[1]) / iters)
    return {k: {"ms_median": statistics.median(v), "ms_min": min(v), "ms_max": max(v), "num_locs": n[k]}
            for k, v in ms.items()}


class StandInGenerator(torch.nn.Module):
    """Seeded Conv3d + BatchNorm3d stand-in of the reference generator's width (nf 20) with its call signature; the
    heads are channels of one 19-channel output.  Not the reference's U-Net: its times are not the reference's."""

    def __init__(self, nf=20):
        super().__init__()
        layers, c = [], 4
        for _ in range(4):
            layers += [torch.nn.Conv3d(c, nf, 3, padding=1), torch.nn.BatchNorm3d(nf), torch.nn.ReLU()]
            c = nf
        self.body = torch.nn.Sequential(*layers)
        self.head = torch.nn.Conv3d(nf, 19, 1)

    def forward(self, inputs, mask, pred_sdf=(True, True), pred_color=True, pred_semantic=True):
        out = self.head(self.body(inputs))
        sdf = inputs[:, :1].to(out.dtype) + 0.3 * torch.tanh(out[:, 1:2])
        return out[:, :1] + 3.0, sdf, torch.tanh(out[:, 2:5]), out[:, 5:19]


def stand_in_losses():
    return types.SimpleNamespace(
        compute_targets=lambda sdf, truncation, flag, known, colors: (sdf.clone(), colors),
        compute_dense_geo_weights=lambda target, input_occ, truncation, w_surf, w_missing: torch.ones_like(target),
        compute_geo_occ_loss=lambda target, occ, known, weight, truncation: Fn.binary_cross_entropy_with_logits(
            occ, (target.abs() < truncation).float(), weight=weight),
        compute_geo_loss=lambda target, unused, sdf, known, weight, logweight: (weight * (sdf - target).abs()).mean())


def time_step(dev, steps, warmup):
    from baseline import ref_loader
    from spsg_b200 import synthetic as S
    from spsg_b200.train_step import ViewGuidedTrainStep, prepare_generator
    torch.backends.cudnn.benchmark = True
    reference = ref_loader.available()
    res = {}
    for autocast in (False, True, False, True):    # alternated; the second of each pair is kept
        torch.manual_seed(7)
        if reference:
            model_util, loss_util = ref_loader.load_module("model"), ref_loader.load_module("loss")
            sys.stdout, keep = open(os.devnull, "w"), sys.stdout
            try:
                model = model_util.Generator(nf_in_geo=1, nf_in_color=4, nf=20, pass_geo_feats=True,
                                             truncation=S.TRUNCATION, max_data_size=S.DIMS_ZYX).to(dev)
            finally:
                sys.stdout = keep
            generator = "reference Generator (baseline/_ref model.py, nf 20, random init)"
        else:
            model, loss_util = StandInGenerator().to(dev), stand_in_losses()
            generator = ("STAND-IN: 4 x (Conv3d 3x3x3 + BatchNorm3d + ReLU) of width 20 + 1x1x1 head, seeded; stand-in "
                         "dense losses -- baseline/_ref is not installed, the reference generator was not measured")
        model = prepare_generator(model.train())
        opt = torch.optim.Adam(model.parameters(), lr=1e-4)
        cw = torch.tensor(S.CLASS_WEIGHTS, dtype=torch.float32, device=dev)
        samples = []
        for k in range(2):
            s = S.make_train_sample([10 + k * B + b for b in range(B)], 1, view_seed=k)
            samples.append({key: torch.from_numpy(v).to(dev) for key, v in s.items()})
        step = ViewGuidedTrainStep(model, loss_util, B, S.DIMS_ZYX, S.WIDTH, S.HEIGHT, cw, max_num_locs_per_sample=640000,
                                   device=dev, autocast_bf16=autocast)
        for i in range(warmup):
            step(dict(samples[i % 2], sdf=samples[i % 2]["sdf"].clone()), optimizer=opt)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(steps):
            loss = step(dict(samples[i % 2], sdf=samples[i % 2]["sdf"].clone()), optimizer=opt)
        b.record()
        torch.cuda.synchronize()
        res["bf16_autocast_ndhwc" if autocast else "fp32_ndhwc"] = {
            "ms_per_step": a.elapsed_time(b) / steps, "steps": steps, "num_locs_last_step": int(step.last["num_locs"]),
            "last_loss": float(loss)}
        del model, opt, step
    res["generator"] = generator
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("head_formats_time: needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    name, limit = card()
    out = {"device": name, "power_limit": limit}
    print("device: %s, power limit %s" % (name, limit), flush=True)
    out["glue_fwd_bwd"] = time_glue(dev, a.rounds, a.iters)
    for k, v in out["glue_fwd_bwd"].items():
        print("glue  %-42s %.3f ms (min %.3f, max %.3f; %d voxels)" % (k, v["ms_median"], v["ms_min"], v["ms_max"],
                                                                         v["num_locs"]), flush=True)
    out["train_step"] = time_step(dev, a.steps, a.warmup)
    print("step generator: %s" % out["train_step"]["generator"])
    for k in ("fp32_ndhwc", "bf16_autocast_ndhwc"):
        v = out["train_step"][k]
        print("step  %-22s %.2f ms per step (%d voxels, loss %.4f)" % (k, v["ms_per_step"], v["num_locs_last_step"],
                                                                     v["last_loss"]), flush=True)
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
