#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric: raycast fwd+bwd rays/s, % of the HBM roofline, train chunks/s (SURVEY.md section 8(d)).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c3|c2|c5]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic input; every timed region below that counts steps runs
exactly K of them:
  c3 (default, BASELINE configs[2])  8 chunks 64x64x128 x 5 views 320x256 (3 276 800 rays): raycast forward with the depth /
                                     colour / 2D-semantic losses fused in, and its backward (voxel gradients)
  c2 (BASELINE configs[1])           one chunk, one view; also reported inside the default line as `c2`
  c5 (BASELINE configs[4])           whole-room 2 cm inference by sliding chunks with multi-view semantic rendering
`value`   rays/s with every input already resident in HBM, the step replayed from a CUDA graph (no host launch latency in
          the device number); distinct input sets are rotated so that consecutive steps never find their data in the
          126 MB L2.
`e2e`     the same metric through the public Python API with HOST buffers: every step copies its voxel tensors, cameras
          and target frames from pinned host memory (copy stream, double-buffered) and reads the loss back.
`roofline`     the dominant kernel (raycast forward) timed with CUDA events on its launch stream (C-ABI timing hook),
               algorithmic bytes per launch (SURVEY.md section 8(d)) over MEASURED_PEAKS.json's HBM copy peak.
`train`        BASELINE configs[3]: the train.py step (reference generator fwd/bwd + 3D losses + three raycasts + 2D losses +
               Adam) on this package's ops, DistributedDataParallel over the ranks (NCCL gradient all-reduce), chunks/s.
`cpu_baseline` the scalar C restatement of the raycast (oracle/, OpenMP over pixels) and BASELINE configs[0] (reference
               generator forward + class-weighted 3D cross-entropy, PyTorch CPU) on the box's host cores.
--impl reference  runs the UNMODIFIED reference: its wrapper (baseline/_ref/.../raycast_rgbd.py) on its CUDA extension
          (oracle/_ref, built from /root/reference where it lies), one view per call as it renders, and its literal
          PyTorch losses; same workload, copy protocol and timing rules.  The reference has no CPU implementation of this
          path, so its arm is its CUDA extension (falls back to the CPU port if the extension is not on the box).
One process per GPU (torchrun sets RANK/LOCAL_RANK/WORLD_SIZE); units are independent chunk x view batches, so ranks shard
them with no data-path collective ("scaling": "weak"); time is the max over ranks.
--dump-outputs DIR  after the timed steps of `value`, rank 0 writes what the last of them returned to its caller as
          DIR/<name>.npy (float32 / float64): the loss terms and the voxel gradients (c2/c3; rows sampled with a fixed seed
          when all of them would exceed DUMP_MAX_BYTES, their indices in voxel_rows.npy), or the room's label histogram
          (c5).  The inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

MAX_LOCS = 640000      # train.py:136 max_num_locs_per_sample (sizes the reference's memsets)
E2E_REPEATS = 3        # timed regions of the end-to-end leg (median reported), both arms
TRAIN_BATCH = 8        # chunks per GPU and step of the train leg (BASELINE configs[2]/[3])
DUMP_MAX_BYTES = 64 * 1000 * 1000  # --dump-outputs: all files together stay below this


def bind_to_gpu_numa_node(dev):
    """Run this rank (and first-touch its pinned host buffers) on the CPUs NVML reports as local to its GPU -- what a
    multi-GPU launcher does; on a two-socket 8-GPU box the host->device copies of the e2e leg otherwise cross the socket
    interconnect.  Best effort: returns a description for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        props = torch.cuda.get_device_properties(dev)
        bus = "%08x:%02x:%02x.0" % (getattr(props, "pci_domain_id", 0), props.pci_bus_id, props.pci_device_id)
        h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return "no NUMA-local CPUs reported"
        os.sched_setaffinity(0, cpus)
        return "bound to %d CPUs local to GPU %s" % (len(cpus), bus)
    except Exception as e:  # NVML missing, container without the affinity syscall, ...
        return "not bound (%s)" % type(e).__name__


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=700)  # ~0.5 s of device-resident c3 steps on a B200
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=["c2", "c3", "c5"])
    ap.add_argument("--sets", type=int, default=0, help="distinct resident input sets to rotate (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the train-step leg (configs[3])")
    ap.add_argument("--no-secondary", action="store_true", help="skip the c2 / un-fused secondary numbers")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs is implemented for --impl ours")
    return args


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 6:
                    self.samples.append(f)
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(s[2 + k].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": int(self.samples[0][1]) if self.samples[0][1].isdigit() else None, "reasons": reasons}


# ---------------------------------------------------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------------------------------------------------

H2D_KEYS = ("locs", "sdf", "color", "normal", "semantic", "view", "intr", "t_depth", "t_color", "t_label")


def make_host_sets(num_sets, B, F, rank):
    """Seeded synthetic chunk batches + cameras + target frames, as pinned host tensors."""
    from spsg_b200 import synthetic as S
    sets = []
    for k in range(num_sets):
        seeds = [1 + rank * 1000 + k * B + b for b in range(B)]
        batch = S.make_batch(seeds)
        view, intr = S.make_views(B, F, seed=rank * 100 + k)
        rng = np.random.default_rng(k + 17 * rank)
        imgs = B * F
        host = {
            "locs": torch.from_numpy(batch["locs"]), "sdf": torch.from_numpy(batch["sdf"]),
            "color": torch.from_numpy(batch["color"]), "normal": torch.from_numpy(batch["normal"]),
            "semantic": torch.from_numpy(batch["semantic"]), "view": torch.from_numpy(view),
            "intr": torch.from_numpy(intr),
            # target frames (2D losses): depth in metres with 5 % holes, colour in [0,1], labels 0..14
            "t_depth": torch.from_numpy(np.where(rng.random((imgs, S.HEIGHT, S.WIDTH)) < 0.05, 0.0,
                                                 rng.uniform(0.8, 1.6, (imgs, S.HEIGHT, S.WIDTH))).astype(np.float32)),
            "t_color": torch.from_numpy(rng.random((imgs, S.HEIGHT, S.WIDTH, 3), dtype=np.float32)),
            "t_label": torch.from_numpy(rng.integers(0, 15, (imgs, S.HEIGHT, S.WIDTH), dtype=np.uint8)),
        }
        sets.append({k2: v.pin_memory() for k2, v in host.items()})
    return sets


def bytes_of(d, keys):
    return int(sum(d[k].numel() * d[k].element_size() for k in keys))


def auto_sets(B, F):
    per_set_mb = 45.0 * B + 14.0 * B * F
    return max(2, int(math.ceil(190.0 / per_set_mb))), per_set_mb


def reduce_max_ms(ms, dev, world):
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms


def timed_replays(graphs, dev, world):
    """One launch of each graph in order, bracketed by barrier + synchronize, CUDA-event time, max over ranks."""
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for graph in graphs:
        graph.replay()
    b.record()
    torch.cuda.synchronize()
    ms = reduce_max_ms(a.elapsed_time(b), dev, world)
    if world > 1:
        dist.barrier()
    return ms


def capture_rotation(step, num_steps, dev, warmup):
    """Warm up, then capture steps 0 .. num_steps-1 (one rotation over the input sets, or its first part) into a CUDA
    graph."""
    for i in range(max(warmup, 3)):
        step(i)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        step(0)
        side.synchronize()
        with torch.cuda.graph(graph, stream=side):
            for i in range(num_steps):
                step(i)
    torch.cuda.current_stream(dev).wait_stream(side)
    for _ in range(2):
        graph.replay()
    torch.cuda.synchronize()
    return graph


def measure_resident(step, num_sets, dev, world, steps, warmup):
    """(ms, graphs) of a device-resident loop of exactly `steps` steps: replays of one captured rotation over the input
    sets, then a graph of the steps left over.  The graphs own the memory of what their steps returned."""
    graph = capture_rotation(step, num_sets, dev, warmup)
    rest = steps % num_sets
    tail = [capture_rotation(step, rest, dev, 0)] if rest else []
    return timed_replays([graph] * (steps // num_sets) + tail, dev, world), [graph] + tail


# ---------------------------------------------------------------------------------------------------------------------
# ours
# ---------------------------------------------------------------------------------------------------------------------

class Ours:
    def __init__(self, dev, rank, B, F, num_sets):
        from spsg_b200 import _native as N
        from spsg_b200 import raycast_rgbd_cuda as rc
        from spsg_b200 import synthetic as S
        from spsg_b200.losses import render_loss_and_voxel_grads, render_with_2d_losses
        from spsg_b200.raycast_rgbd import RaycastRGBD
        self.N, self.rc, self.S, self.render, self.render_pair = N, rc, S, render_with_2d_losses, render_loss_and_voxel_grads
        self.dev, self.B, self.F, self.num_sets = dev, B, F, num_sets
        self.host = make_host_sets(num_sets, B, F, rank)
        self.rays = B * F * S.WIDTH * S.HEIGHT
        self.devsets, self.mods, self.grads = [], [], []
        for h in self.host:
            d = {k: v.to(dev, non_blocking=True) for k, v in h.items()}
            self.devsets.append(d)
            self.mods.append(RaycastRGBD(B, S.DIMS_ZYX, S.WIDTH, S.HEIGHT, S.DEPTH_MIN, S.DEPTH_MAX, S.THRESH_SAMPLE_DIST,
                                         S.RAY_INCREMENT, max_num_frames=F, max_num_locs_per_sample=MAX_LOCS, device=dev))
            g = torch.Generator(device=dev).manual_seed(5)
            self.grads.append([torch.randn(s, device=dev, generator=g) for s in
                               ((B * F, S.HEIGHT, S.WIDTH, 3), (B * F, S.HEIGHT, S.WIDTH), (B * F, S.HEIGHT, S.WIDTH, 3),
                                (B * F, S.HEIGHT, S.WIDTH, 14))])
        self.nv = int(np.mean([d["locs"].shape[0] for d in self.devsets]))
        self.cw = torch.tensor(S.CLASS_WEIGHTS, dtype=torch.float32, device=dev)
        self.loss_sink = torch.zeros((), device=dev)
        self.returned = {}

    def step_fused(self, i):
        """forward with the three 2D losses fused in + backward from the scalar loss (the north-star path)."""
        S = self.S
        k = i % self.num_sets
        d, m = self.devsets[k], self.mods[k]
        # the two native calls of spsg_b200.losses (spsg_raycast_forward_loss + spsg_raycast_backward_loss) without the
        # autograd wrapper: voxel gradients land in the module's d_* rows, the loss in loss_out[3]
        loss_out, grads = self.render_pair(m, d["locs"], d["sdf"], d["color"], d["normal"], d["semantic"], d["view"],
                                           d["intr"], images_depth=d["t_depth"], images_color=d["t_color"],
                                           target2d_label=d["t_label"], weight_semantic_class=self.cw, voxelsize=S.VOXELSIZE)
        self.loss_sink.copy_(loss_out[3])
        self.returned[k] = (loss_out, grads)  # when captured: the tensors every replay of this step writes

    def last_outputs(self, steps):
        """What the last of `steps` fused steps returned: its loss_out and voxel gradients, as numpy arrays."""
        loss_out, grads = self.returned[(steps - 1) % self.num_sets]
        out = {"loss_out": loss_out}
        out.update(zip(("d_sdf", "d_color", "d_normal", "d_semantic"), grads))
        return {k: v.detach().cpu().numpy() for k, v in out.items()}

    def step_unfused(self, i):
        """forward + backward with upstream gradient images (the reference op boundary)."""
        S, rc, B, F = self.S, self.rc, self.B, self.F
        k = i % self.num_sets
        d, m, g = self.devsets[k], self.mods[k], self.grads[k]
        n = d["locs"].shape[0]
        opts = [S.WIDTH, S.HEIGHT, S.DEPTH_MIN, S.DEPTH_MAX, S.THRESH_SAMPLE_DIST, S.RAY_INCREMENT, 64, 64, 128]
        rc.forward(m.sparse_mapping, d["locs"], d["sdf"], d["color"], d["normal"], d["semantic"], d["view"],
                   m.image_color, m.image_depth, m.image_normal, m.image_semantic, m.mapping3dto2d,
                   m.mapping3dto2d_num, d["intr"], opts, views_per_chunk=F, build_index=True,
                   clear_grads=(m.d_color, m.d_depth, m.d_normal, m.d_semantic))
        rc.backward(g[0], g[1], g[2], g[3], m.sparse_mapping, m.mapping3dto2d, m.mapping3dto2d_num,
                    [B, 64, 64, 128, n], m.d_color, m.d_depth, m.d_normal, m.d_semantic, views_per_chunk=F,
                    grads_cleared=True)

    def e2e(self, world, steps, warmup):
        """End to end through the public API with HOST inputs: every step copies its voxel tensors, cameras and target
        frames from pinned host memory (on a copy stream, double-buffered so that step i+1's copy overlaps step i's
        kernels -- what a training loop's prefetcher does), renders + losses + backward, and reads the loss back."""
        S, render, mods, host, cw, dev = self.S, self.render, self.mods, self.host, self.cw, self.dev
        num_sets = len(host)
        result = torch.zeros((), pin_memory=True)
        copy_stream = torch.cuda.Stream(device=dev)
        main = torch.cuda.current_stream(dev)
        # The loader's voxel rows are the reference's (N,4) int64; what crosses PCIe is one uint32 cell index per row,
        # packed on the host by this package (spsg_pack_locs_host, OpenMP over the rank's CPUs) EVERY step, inside the
        # timed region, straight into the step's pinned staging buffer.
        packed = [pack_host(h, narrow_locs=True) for h in host]
        cap = max(b.numel() for b, _ in packed)
        slots = [torch.empty(cap, dtype=torch.uint8, device=dev) for _ in range(2)]
        copied = [torch.cuda.Event() for _ in range(2)]
        consumed = [torch.cuda.Event() for _ in range(2)]
        read_by_copy = [torch.cuda.Event() for _ in range(num_sets)]  # last copy out of staging buffer k
        staged_locs = [slot_views(b, {"locs": f["locs"]})["locs"] for b, f in packed]
        pack_threads = max(1, min(16, len(os.sched_getaffinity(0)) // max(1, world)))  # the ranks of a node share its CPUs

        def issue_copy(i):
            slot, k = i % 2, i % num_sets
            buf = packed[k][0]
            read_by_copy[k].synchronize()  # (a loader must not rewrite a staging buffer a copy is still reading)
            self.rc.pack_locs_host(host[k]["locs"], self.B, S.DIMS_ZYX, out=staged_locs[k], threads=pack_threads)
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[slot])  # the step that last used this slot is done with it
                slots[slot][:buf.numel()].copy_(buf, non_blocking=True)
                copied[slot].record(copy_stream)
                read_by_copy[k].record(copy_stream)

        view_cache = {}

        def views(i):
            key = (i % 2, i % num_sets)
            if key not in view_cache:
                view_cache[key] = slot_views(slots[key[0]], packed[key[1]][1])
            return view_cache[key]

        def step(i, last):
            slot, m = i % 2, mods[i % num_sets]
            if not last:
                issue_copy(i + 1)
            main.wait_event(copied[slot])
            d = views(i)
            sdf = d["sdf"].detach().requires_grad_(True)  # fresh leaves every step
            col = d["color"].detach().requires_grad_(True)
            sem = d["semantic"].detach().requires_grad_(True)
            total, _, _ = render(m, d["locs"], sdf, col, d["normal"], sem, d["view"], d["intr"],
                                 images_depth=d["t_depth"], images_color=d["t_color"], target2d_label=d["t_label"],
                                 weight_semantic_class=cw, voxelsize=S.VOXELSIZE)
            total.backward()
            consumed[slot].record(main)
            result.copy_(total.detach(), non_blocking=True)

        def run(n):
            for e in consumed:
                e.record(main)
            issue_copy(0)
            for i in range(n):
                step(i, i == n - 1)

        ms = e2e_protocol(run, steps, warmup, dev, world)

        # The same bytes with nothing behind them: every rank copies its packed buffer at the same time (max over ranks).
        # e2e above cannot be faster than this; with several GPUs it shows what the host's memory system and PCIe
        # topology give each GPU when all of them pull at once.
        def copies(n):
            for i in range(n):
                buf = packed[i % num_sets][0]
                slots[i % 2][:buf.numel()].copy_(buf, non_blocking=True)
        ms_copy = e2e_protocol(copies, 10, 3, dev, world) / 10
        staged = int(sum(f[1] for f in packed[0][1].values()))
        return ms, float(result), {"ms_per_step": ms_copy, "gb_per_s_per_gpu": packed[0][0].numel() / (ms_copy * 1e-3) / 1e9,
                                   "h2d_bytes_per_step": staged, "host_pack_threads": pack_threads}

    def e2e_device_flow(self, world, steps, warmup):
        """The training data flow: the voxel tensors never come from the host -- the generator leaves dense heads (SDF,
        colour, 14 logits per cell) in HBM -- and only the step's frames (depth, colour, labels, cameras) do.  Per step:
        host -> device copy of the frames (pinned, copy stream, two slots), then on the device the stream-compaction
        sparsify of the heads (train.py:494-509; its one host read of N included), the sparse normals (loss.py:285-306),
        the fused raycast + 2D losses, the backward down to dense head gradients, and the loss read back."""
        from spsg_b200 import normals as NRM
        from spsg_b200 import sparsify as SP
        S, render, mods, host, cw, dev, B, F = self.S, self.render, self.mods, self.host, self.cw, self.dev, self.B, self.F
        num_sets = len(host)
        dz, dy, dx = S.DIMS_ZYX
        heads = []
        for h in host:  # dense heads of every input set, made once: they are the generator's (resident) output
            locs = h["locs"].to(dev)
            idx = (locs[:, 3], locs[:, 0], locs[:, 1], locs[:, 2])
            sdf = torch.full((B, dz, dy, dx), 2.0 * S.TRUNCATION, device=dev)
            sdf[idx] = h["sdf"].to(dev)[:, 0]
            col = torch.zeros(B, dz, dy, dx, 3, device=dev)
            col[idx] = h["color"].to(dev)
            sem = torch.zeros(B, dz, dy, dx, 14, device=dev)
            sem[idx] = h["semantic"].to(dev)
            heads.append((sdf.unsqueeze(1).contiguous(), col.permute(0, 4, 1, 2, 3).contiguous(),
                          sem.permute(0, 4, 1, 2, 3).contiguous()))
        keys = ("view", "intr", "t_depth", "t_color", "t_label")
        packed = [pack_host(h, keys) for h in host]
        cap = max(b.numel() for b, _ in packed)
        slots = [torch.empty(cap, dtype=torch.uint8, device=dev) for _ in range(2)]
        copied = [torch.cuda.Event() for _ in range(2)]
        consumed = [torch.cuda.Event() for _ in range(2)]
        copy_stream = torch.cuda.Stream(device=dev)
        main = torch.cuda.current_stream(dev)
        result = torch.zeros((), pin_memory=True)

        def issue_copy(i):
            slot, (buf, _) = i % 2, packed[i % num_sets]
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[slot])
                slots[slot][:buf.numel()].copy_(buf, non_blocking=True)
                copied[slot].record(copy_stream)

        def step(i, last):
            slot, k = i % 2, i % num_sets
            if not last:
                issue_copy(i + 1)
            main.wait_event(copied[slot])
            d = slot_views(slots[slot], packed[k][1])
            sdf, col, sem = (t.detach().requires_grad_(True) for t in heads[k])
            locs, v_sdf, v_col, v_sem = SP.sparsify_predictions(sdf, S.TRUNCATION, None, col, sem, raycaster=mods[k])
            nrm = NRM.compute_normals_sparse(locs, v_sdf, S.DIMS_ZYX, transform=torch.inverse(d["view"][::F]), num_chunks=B)
            total, _, _ = render(mods[k], locs, v_sdf, v_col, nrm, v_sem, d["view"], d["intr"], images_depth=d["t_depth"],
                                 images_color=d["t_color"], target2d_label=d["t_label"], weight_semantic_class=cw,
                                 voxelsize=S.VOXELSIZE)
            total.backward()
            consumed[slot].record(main)
            result.copy_(total.detach(), non_blocking=True)

        def run(n):
            for e in consumed:
                e.record(main)
            issue_copy(0)
            for i in range(n):
                step(i, i == n - 1)

        ms = e2e_protocol(run, steps, warmup, dev, world)
        return ms, float(result), bytes_of(host[0], keys)

    def roofline(self, steps, fused):
        """Dominant kernel (raycast forward) alone: CUDA events around each launch on its stream, inputs rotated."""
        N = self.N
        N.timing_read(0), N.timing_read(1)
        N.timing_enable(True)
        for i in range(steps):
            (self.step_fused if fused else self.step_unfused)(i)
        torch.cuda.synchronize()
        N.timing_enable(False)
        f_ms, f_n = N.timing_read(0)
        g_ms, g_n = N.timing_read(1)
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.isfile(peaks_path):
            peak, which = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            peak, which = 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"
        # forward: locs 32 B + payload 84 B per voxel in, 84 B per pixel out (+ 17 B of targets per pixel when fused)
        alg_bytes = 116 * self.nv + (84 + (17 if fused else 0)) * self.rays
        us = f_ms / max(f_n, 1) * 1e3
        achieved = alg_bytes / (us * 1e-6) / 1e9 if us > 0 else 0.0
        traffic, traffic_src = ncu_traffic("c%d" % (3 if self.B * self.F > 1 else 2))
        return {"bound": "hbm", "kernel": "raycast_forward_kernel" + ("<loss>" if fused else ""),
                "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                "traffic": traffic, "traffic_source": traffic_src, "peak_source": which,
                "algorithmic_bytes_per_launch": alg_bytes, "kernel_us": round(us, 2),
                "backward_gather_us": round(g_ms / max(g_n, 1) * 1e3, 2),
                "note": "not HBM-bound (traffic ~ algorithmic bytes): instruction issue / per-warp latency, see DESIGN.md "
                        "section 5 and profiles/README.md"}


def dump_outputs(path, arrays):
    """Write each array as path/<name>.npy (float32 stays float32; integers, so that counts stay exact, and everything
    else become float64).  When the per-voxel arrays (those with the most rows) would take the files past DUMP_MAX_BYTES,
    the same fixed, seeded sample of their rows is written and voxel_rows.npy holds its indices."""
    arrays = {k: np.asarray(v) for k, v in arrays.items()}
    arrays = {k: a.astype(np.float32 if a.dtype == np.float32 else np.float64) for k, a in arrays.items()}
    rows = max(a.shape[0] if a.ndim else 0 for a in arrays.values())
    per_voxel = [k for k, a in arrays.items() if a.ndim and a.shape[0] == rows]
    total = sum(a.nbytes for a in arrays.values())
    budget = DUMP_MAX_BYTES - 256 * (len(arrays) + 1)  # .npy headers
    if total > budget:
        row_bytes = sum(arrays[k].nbytes // rows for k in per_voxel) + 8  # + its float64 index
        keep = (budget - (total - sum(arrays[k].nbytes for k in per_voxel))) // row_bytes
        sel = np.sort(np.random.default_rng(0).choice(rows, size=keep, replace=False))
        arrays = dict(arrays, voxel_rows=sel.astype(np.float64), **{k: arrays[k][sel] for k in per_voxel})
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


def ncu_traffic(workload):
    """dram__bytes_read.sum + dram__bytes_write.sum of the forward kernel per launch, from the committed `ncu --set full`
    capture listed in profiles/ncu_traffic.json (written by tools/ncu_summary.py --traffic); None when there is none."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        entry = json.load(open(path))[workload]
        return float(entry["dram_bytes_per_launch"]), "profiles/%s (%s)" % (entry["summary"], entry["kernel"])
    except Exception:
        return None, "no committed ncu capture for this workload"


def pack_host(h, keys=H2D_KEYS, narrow_locs=False):
    """One pinned host buffer per input set (256-byte aligned fields, what a loader thread would hand over).
    narrow_locs: the field of the voxel rows holds one uint32 cell index per row (4 bytes instead of the reference's 32); it
    is left unwritten here -- the caller packs the loader's int64 rows into it every step (spsg_pack_locs_host)."""
    off, fields = 0, {}
    for k in keys:
        if k == "locs" and narrow_locs:
            dtype, shape = torch.int32, (h[k].shape[0],)
            nbytes = 4 * h[k].shape[0]
        else:
            dtype, shape = h[k].dtype, tuple(h[k].shape)
            nbytes = h[k].numel() * h[k].element_size()
        fields[k] = (off, nbytes, dtype, shape)
        off += (nbytes + 255) // 256 * 256
    buf = torch.empty(off, dtype=torch.uint8).pin_memory()
    for k, (o, nbytes, dtype, shape) in fields.items():
        if not (k == "locs" and narrow_locs):
            buf[o:o + nbytes].view(dtype).view(shape).copy_(h[k])
    return buf, fields


def slot_views(slot, fields):
    return {k: slot[off:off + nbytes].view(dtype).view(shape) for k, (off, nbytes, dtype, shape) in fields.items()}


def e2e_protocol(run, steps, warmup, dev, world):
    """Warm up, then the median of E2E_REPEATS timed regions of `steps` steps (max over ranks each)."""
    run(max(3, warmup))
    times = []
    for _ in range(E2E_REPEATS):  # host-side jitter is of the order of the step: median of a few timed regions
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        run(steps)
        b.record()
        torch.cuda.synchronize()
        times.append(reduce_max_ms(a.elapsed_time(b), dev, world))
    return float(np.median(times))


# ---------------------------------------------------------------------------------------------------------------------
# train step (BASELINE configs[3]) and CPU baselines
# ---------------------------------------------------------------------------------------------------------------------

def train_leg(impl, dev, rank, world, local, steps=8, warmup=3, layout="ncdhw"):
    """chunks/s of the train.py step under DistributedDataParallel (one rank per GPU, NCCL all-reduce of the generator's
    gradients); impl "ours" = spsg_b200.train_step on this package's ops, "reference" = the reference's loop body, wrapper,
    losses and CUDA extension (baseline/ref_train_step.py)."""
    from baseline import ref_loader
    from spsg_b200 import synthetic as S
    if not ref_loader.available():
        return {"unavailable": "baseline/_ref (reference model.py / loss.py) is not installed on this box"}
    model_util = ref_loader.load_module("model")
    loss_util = ref_loader.load_module("loss")
    torch.backends.cudnn.benchmark = True  # train.py:122
    torch.manual_seed(7)
    sys.stdout, keep = open(os.devnull, "w"), sys.stdout  # the reference's Generator prints its parameter counts
    try:
        model = model_util.Generator(nf_in_geo=1, nf_in_color=4, nf=20, pass_geo_feats=True, truncation=S.TRUNCATION,
                                     max_data_size=S.DIMS_ZYX).to(dev)  # train.py:153-156 defaults
    finally:
        sys.stdout = keep
    model.train()
    if layout == "ndhwc":
        from spsg_b200.train_step import prepare_generator
        model = prepare_generator(model)  # memory format only: same modules, same arithmetic
    params = sum(p.numel() for p in model.parameters())
    net = model
    if world > 1:
        net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local], bucket_cap_mb=25)
    opt = torch.optim.Adam(model.parameters(), lr=1e-4)  # train.py:157
    cw = torch.tensor(S.CLASS_WEIGHTS, dtype=torch.float32, device=dev)
    samples = []
    for k in range(2):
        s = S.make_train_sample([10 + rank * 100 + k * TRAIN_BATCH + b for b in range(TRAIN_BATCH)], 1, view_seed=rank * 10 + k)
        samples.append({key: torch.from_numpy(v).to(dev) for key, v in s.items()})
    if impl == "ours":
        from spsg_b200.train_step import ViewGuidedTrainStep
        step = ViewGuidedTrainStep(net, loss_util, TRAIN_BATCH, S.DIMS_ZYX, S.WIDTH, S.HEIGHT, cw,
                                   max_num_locs_per_sample=MAX_LOCS, device=dev)
    else:
        from baseline.ref_train_step import RefTrainStep
        step = RefTrainStep(net, TRAIN_BATCH, S.DIMS_ZYX, S.WIDTH, S.HEIGHT, cw, native="reference",
                            max_num_locs_per_sample=MAX_LOCS)

    def one(i):
        s = samples[i % 2]
        # the reference's compute_targets clamps the target SDF in place (data_util.py:187-190): hand it a copy, like a
        # dataloader's fresh batch
        return step(dict(s, sdf=s["sdf"].clone()), optimizer=opt)

    for i in range(warmup):
        one(i)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(steps):
        loss = one(i)
    b.record()
    torch.cuda.synchronize()
    ms = reduce_max_ms(a.elapsed_time(b), dev, world)
    return {"chunks_per_s": world * TRAIN_BATCH * steps / (ms * 1e-3), "unit": "chunks/s", "ms_per_step": ms / steps,
            "steps": steps, "chunks_per_gpu_per_step": TRAIN_BATCH, "views_per_chunk": 1,
            "generator_parameters": params, "num_locs_last_step": int(step.last.get("num_locs", -1)),
            "last_loss": float(loss),
            "generator_layout": "channels_last_3d (NDHWC) parameters and activations" if layout == "ndhwc" else
                                "PyTorch default (NCDHW)",
            "step": ("spsg_b200.train_step.ViewGuidedTrainStep: reference Generator (baseline/_ref model.py, random init) "
                     "fwd/bwd + its dense 3D losses + sparsify / normals / 3 raycasts / fused 2D losses of this package + Adam"
                     if impl == "ours" else
                     "baseline/ref_train_step.py: train.py:399-757 loop body on the reference's Generator, loss module, "
                     "raycast_rgbd.py wrapper and CUDA extension + Adam"),
            "collective": ("DistributedDataParallel, NCCL all-reduce of %.1f MB of gradients in one bucket, overlapped with "
                           "backward" % (params * 4 / 1e6)) if world > 1 else "none (1 rank)"}


def cpu_raycast_baseline(seconds=12.0):
    """Scalar C restatement of the raycast fwd+bwd (oracle/raycast_oracle.c), OpenMP over pixels, host cores."""
    from oracle import oracle as O
    from spsg_b200 import synthetic as S
    threads = O.max_threads()
    b = S.make_batch([1])
    view, intr = S.make_views(1, 1, seed=0)
    n = b["locs"].shape[0]
    p = O.make_params(S.DIMS_ZYX, S.WIDTH, S.HEIGHT, S.DEPTH_MIN, S.DEPTH_MAX, S.THRESH_SAMPLE_DIST, S.RAY_INCREMENT, 1,
                      1, 64, n)
    rng = np.random.default_rng(0)
    g = None
    t0, steps = time.perf_counter(), 0
    while True:
        sm = O.build_index(b["locs"], 1, S.DIMS_ZYX)
        out = O.raycast_forward(p, sm, b["sdf"], b["color"], b["normal"], b["semantic"], view, intr, threads=threads)
        if g is None:
            g = [rng.standard_normal(out[k].shape).astype(np.float32) for k in ("color", "depth", "normal", "semantic")]
        O.raycast_backward(p, *g, sm, out["mapping3dto2d"], out["mapping3dto2d_num"])
        steps += 1
        dt = time.perf_counter() - t0
        if dt > seconds or steps >= 400:
            break
    rays = S.WIDTH * S.HEIGHT * steps
    return {"value": rays / dt, "unit": "rays/s", "cores": threads, "kind": "port",
            "sample": "%d fwd+bwd steps of one chunk x one 320x256 view (the c3 batch is 40 such images) in %.1f s; forward "
                      "OpenMP over pixels on %d threads, backward scalar" % (steps, dt, threads)}


def cpu_generator_baseline(max_seconds=25.0):
    """BASELINE configs[0]: reference Generator forward + class-weighted 3D semantic cross-entropy on one synthetic
    64x64x128 chunk, batch 1, PyTorch CPU, default intra-op threads (2D losses off)."""
    from baseline import ref_loader
    from spsg_b200 import synthetic as S
    if not ref_loader.available():
        return {"unavailable": "baseline/_ref is not installed on this box"}
    model_util = ref_loader.load_module("model")
    torch.manual_seed(7)
    sys.stdout, keep = open(os.devnull, "w"), sys.stdout
    try:
        model = model_util.Generator(nf_in_geo=1, nf_in_color=4, nf=20, pass_geo_feats=True, truncation=S.TRUNCATION,
                                     max_data_size=S.DIMS_ZYX)
    finally:
        sys.stdout = keep
    model.eval()
    s = S.make_train_sample([3], 1)
    inputs, mask = torch.from_numpy(s["input"]), torch.from_numpy(s["mask"])
    label = torch.from_numpy(s["semantics"])[:, 0]
    cw = torch.tensor(S.CLASS_WEIGHTS, dtype=torch.float32)
    times_f, times_l = [], []
    t_all = time.perf_counter()
    with torch.no_grad():
        for it in range(4):
            t0 = time.perf_counter()
            _, out_sdf, _, out_sem = model(inputs.clone(), mask, pred_sdf=[True, True], pred_color=True, pred_semantic=True)
            t1 = time.perf_counter()
            # train.py:494-509, 736-741: logits and labels at the predicted voxels, labelled ones only
            locs = torch.nonzero(torch.abs(out_sdf[:, 0]) < S.TRUNCATION)
            logits = out_sem[locs[:, 0], :, locs[:, 1], locs[:, 2], locs[:, 3]]
            tgt = label[locs[:, 0], locs[:, 1], locs[:, 2], locs[:, 3]]
            keep_rows = tgt < 14
            loss = torch.nn.functional.cross_entropy(logits[keep_rows], tgt[keep_rows], weight=cw) if keep_rows.any() \
                else torch.zeros(())
            t2 = time.perf_counter()
            if it > 0 or time.perf_counter() - t_all > max_seconds:
                times_f.append(t1 - t0)
                times_l.append(t2 - t1)
            if time.perf_counter() - t_all > max_seconds:
                break
    f, l = float(np.median(times_f)), float(np.median(times_l))
    return {"value": 1.0 / (f + l), "unit": "chunks/s", "cores": torch.get_num_threads(), "kind": "reference",
            "generator_forward_s": f, "semantic_3d_ce_s": l, "voxels_in_loss": int(keep_rows.sum()),
            "last_loss": float(loss),
            "sample": "configs[0]: reference model.Generator (nf 20, random init) forward + class-weighted 3D cross-entropy "
                      "on one synthetic 64x64x128 chunk, batch 1, PyTorch CPU with %d intra-op threads, median of %d passes"
                      % (torch.get_num_threads(), len(times_f))}


# ---------------------------------------------------------------------------------------------------------------------
# reference arm
# ---------------------------------------------------------------------------------------------------------------------

class Reference:
    """The unmodified reference: its Python wrapper (baseline/_ref) when installed -- else its native entry points in the
    wrapper's call order (oracle/ref_driver.py) -- on its CUDA extension; one view per call, as it renders."""

    def __init__(self, dev, rank, B, F, num_sets):
        from baseline import ref_loader
        from oracle import losses_ref as R
        from oracle import ref_driver
        from spsg_b200 import synthetic as S
        self.S, self.R, self.dev, self.B, self.F, self.num_sets = S, R, dev, B, F, num_sets
        self.host = make_host_sets(num_sets, B, F, rank)
        self.rays = B * F * S.WIDTH * S.HEIGHT
        self.cw = torch.tensor(S.CLASS_WEIGHTS, dtype=torch.float32, device=dev)
        self.through_wrapper = ref_loader.available()
        if self.through_wrapper:
            wrapper = ref_loader.load_wrapper("reference")
            self.ref = wrapper.RaycastRGBD(B, S.DIMS_ZYX, S.WIDTH, S.HEIGHT, S.DEPTH_MIN, S.DEPTH_MAX, S.THRESH_SAMPLE_DIST,
                                           S.RAY_INCREMENT, max_num_locs_per_sample=MAX_LOCS)
        else:
            self.ref = ref_driver.RefRaycaster(B, S.DIMS_ZYX, S.WIDTH, S.HEIGHT, S.DEPTH_MIN, S.DEPTH_MAX,
                                               S.THRESH_SAMPLE_DIST, S.RAY_INCREMENT, MAX_LOCS, 64, device=dev)
        self.devsets = [self.split_views({k: v.to(dev) for k, v in h.items()}) for h in self.host]
        g = torch.Generator(device=dev).manual_seed(5)
        self.grads = [torch.randn(s, device=dev, generator=g) for s in
                      ((B, S.HEIGHT, S.WIDTH, 3), (B, S.HEIGHT, S.WIDTH), (B, S.HEIGHT, S.WIDTH, 3), (B, S.HEIGHT, S.WIDTH, 14))]
        self.nv = int(np.mean([d["locs"].shape[0] for d in self.devsets]))

    def split_views(self, d):
        """Per-view camera and target tensors (image i = chunk i // F, view i % F), made once per input set: the reference
        takes one view per chunk and call."""
        B, F = self.B, self.F
        sel = [torch.arange(B, device=d["view"].device) * F + f for f in range(F)]
        for k in ("view", "intr", "t_depth", "t_color", "t_label"):
            d[k + "_v"] = [d[k][s].contiguous() for s in sel]
        return d

    def render(self, d, f, sdf, col, sem):
        if self.through_wrapper:
            return self.ref(d["locs"], sdf, col, d["normal"], sem, d["view_v"][f], d["intr_v"][f])
        return self.ref.forward(d["locs"], sdf, col, d["normal"], sem, d["view_v"][f], d["intr_v"][f])

    def step_resident(self, i):
        """F x (forward + backward with upstream gradient images): the reference op boundary."""
        d = self.devsets[i % self.num_sets]
        for f in range(self.F):
            if self.through_wrapper:
                sdf, col, sem = (d[k].detach().requires_grad_(True) for k in ("sdf", "color", "semantic"))
                out = self.render(d, f, sdf, col, sem)
                torch.autograd.backward(out, self.grads)
            else:
                self.render(d, f, d["sdf"], d["color"], d["semantic"])
                self.ref.backward(*self.grads)

    def losses(self, d, f, out):
        S, R = self.S, self.R
        label = d["t_label_v"][f].unsqueeze(-1)
        return R.depth_l1_loss(out[1], d["t_depth_v"][f].unsqueeze(1), S.VOXELSIZE) + \
            R.compute_2dcolor_loss(out[0], d["t_color_v"][f], None) + R.semantic_2d_ce_loss(out[3], label, self.cw)

    def step_fused_equivalent(self, d):
        """F x (render + the literal depth / colour / 2D-semantic losses + backward to the voxels), train.py:626-643,744-757."""
        total = None
        for f in range(self.F):
            sdf, col, sem = (d[k].detach().requires_grad_(True) for k in ("sdf", "color", "semantic"))
            if self.through_wrapper:
                out = self.render(d, f, sdf, col, sem)
                loss = self.losses(d, f, out)
                loss.backward()
            else:
                out = self.render(d, f, sdf, col, sem)
                imgs = [o.detach().clone().requires_grad_(True) for o in out]
                loss = self.losses(d, f, imgs)
                loss.backward()
                self.ref.backward(imgs[0].grad, imgs[1].grad, torch.zeros_like(imgs[2]), imgs[3].grad)
            total = loss.detach() if total is None else total + loss.detach()
        return total

    def e2e(self, world, steps, warmup):
        """Same protocol as the product arm: one packed pinned buffer per set, copy stream, two device slots."""
        dev, num_sets = self.dev, self.num_sets
        result = torch.zeros((), pin_memory=True)
        copy_stream = torch.cuda.Stream(device=dev)
        main = torch.cuda.current_stream(dev)
        packed = [pack_host(h) for h in self.host]
        cap = max(b.numel() for b, _ in packed)
        slots = [torch.empty(cap, dtype=torch.uint8, device=dev) for _ in range(2)]
        copied = [torch.cuda.Event() for _ in range(2)]
        consumed = [torch.cuda.Event() for _ in range(2)]

        def issue_copy(i):
            slot, (buf, _) = i % 2, packed[i % num_sets]
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[slot])
                slots[slot][:buf.numel()].copy_(buf, non_blocking=True)
                copied[slot].record(copy_stream)

        def step(i, last):
            slot = i % 2
            if not last:
                issue_copy(i + 1)
            main.wait_event(copied[slot])
            d = self.split_views(slot_views(slots[slot], packed[i % num_sets][1]))
            total = self.step_fused_equivalent(d)
            consumed[slot].record(main)
            result.copy_(total.reshape(()), non_blocking=True)

        def run(n):
            for e in consumed:
                e.record(main)
            issue_copy(0)
            for i in range(n):
                step(i, i == n - 1)

        return e2e_protocol(run, steps, warmup, dev, world)

    def resident(self, world, steps, warmup):
        for i in range(max(3, warmup)):
            self.step_resident(i)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(steps):
            self.step_resident(i)
        b.record()
        torch.cuda.synchronize()
        return reduce_max_ms(a.elapsed_time(b), self.dev, world)


# ---------------------------------------------------------------------------------------------------------------------
# whole-room workload (BASELINE configs[4])
# ---------------------------------------------------------------------------------------------------------------------

def run_room(args, dev, rank, world, base):
    from spsg_b200 import parallel as P
    from spsg_b200 import room as R
    dims = (128, 256, 320)
    room = R.synthetic_room_sdf(dims, dev)
    predict = R.synthetic_predictor(room)
    kw = dict(views_per_chunk=5, chunks_per_launch=8, rank=rank, world=world)
    windows = R.chunk_windows(dims)
    mine = [windows[i] for i in P.shard_round_robin(len(windows), rank, world)]
    predict.prepare_groups([mine[s:s + 8] for s in range(0, len(mine), 8)], (64, 64))
    for _ in range(max(1, min(args.warmup, 3))):
        out = R.render_room(predict, dims, dev, **kw)
    sampler = ClockSampler(dev.index)
    sampler.start()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    reps = args.steps
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        out = R.render_room(predict, dims, dev, **kw)
    b.record()
    torch.cuda.synchronize()
    sampler.stop_flag = True
    ms = reduce_max_ms(a.elapsed_time(b), dev, world)
    rays = out["rays"]
    if world > 1:
        t = torch.tensor([float(rays)], device=dev, dtype=torch.float64)
        dist.all_reduce(t)
        rays = float(t.item())
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"label_hist": out["label_hist"]})
        value = rays * reps / (ms * 1e-3)
        print(json.dumps(dict(base, value=value, steps=reps, ms_per_step=ms / reps, clocks=sampler.summary(),
                              e2e={"value": value, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 15 * 8,
                                   "note": "a step is one whole room from the generator's dense heads (resident, as a generator "
                                           "leaves them) to label maps + histogram read back; windows dealt round-robin to ranks"},
                              gpu_launches=None, roofline=None)))


# ---------------------------------------------------------------------------------------------------------------------

def main():
    args = parse_args()
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: this implementation has no CPU path")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    numa = bind_to_gpu_numa_node(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from spsg_b200 import synthetic as S
    if args.workload == "c5":
        config = {"workload": "c5: synthetic room 128x256x320 split into 64x64 windows (stride 32), 5 views 320x256 per window, "
                              "sparsify + normals + raycast + label maps, windows sharded over ranks",
                  "parallelism": "dp%d (windows round-robin)" % world,
                  "l2": "one room's windows and images (> 1 GB) stream through between repeats"}
        base = {"metric": "raycast rays/s (whole-room rendering)", "unit": "rays/s", "n_gpus": world, "warmup": args.warmup,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config}
        if args.impl == "reference":
            if rank == 0:
                print(json.dumps({"impl": "reference", "unavailable": "the reference's test_scene_as_chunks.py renders nothing "
                                  "(SURVEY.md section 8 (iv)): there is no reference arm for c5"}))
        else:
            run_room(args, dev, rank, world, base)
        if world > 1:
            dist.destroy_process_group()
        return
    B, F = (1, 1) if args.workload == "c2" else (8, 5)
    auto, per_set_mb = auto_sets(B, F)
    num_sets = args.sets or auto
    config = {"workload": "%s: %d chunk(s) 64x64x128 x %d view(s) 320x256, depth+colour+normal+semantic renderings, forward "
                          "with fused depth/colour/2D-semantic losses + backward" % (args.workload, B, F),
              "chunks_per_step": B, "views_per_chunk": F, "rays_per_step": B * F * S.WIDTH * S.HEIGHT,
              "max_num_locs_per_sample": MAX_LOCS, "parallelism": "dp%d (independent chunk x view batches)" % world,
              "host_affinity": numa,
              "l2": "rotating %d distinct resident input sets (~%d MB > 126 MB L2) between timed steps"
                    % (num_sets, int(per_set_mb * num_sets))}
    base = {"metric": "raycast fwd+bwd rays/s", "unit": "rays/s", "n_gpus": world, "warmup": args.warmup,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config}

    if args.impl == "reference":
        from oracle import ref_driver
        if ref_driver.available():
            r = Reference(dev, rank, B, F, num_sets)
            steps = args.steps
            sampler = ClockSampler(dev.index)
            sampler.start()
            ms = r.resident(world, steps, args.warmup)
            sampler.stop_flag = True
            ms_e2e = r.e2e(world, steps, min(args.warmup, 3))
            value = world * r.rays * steps / (ms * 1e-3)
            e2e = world * r.rays * steps / (ms_e2e * 1e-3)
            line = dict(base, impl="reference", value=value, steps=steps, ms_per_step=ms / steps,
                        clocks=sampler.summary(), gpu_launches=0,
                        e2e={"value": e2e, "unit": "rays/s", "h2d_bytes_per_step": bytes_of(r.host[0], H2D_KEYS),
                             "d2h_bytes_per_step": 4, "steps": steps, "ms_per_step": ms_e2e / steps,
                             "api": "%s + literal depth/colour/semantic losses + backward, %d call(s) per step (one view "
                                    "per chunk and call); inputs from one packed pinned buffer on a copy stream "
                                    "(double-buffered), median of %d timed regions -- the product arm's protocol"
                                    % ("reference RaycastRGBD wrapper (baseline/_ref)" if r.through_wrapper else
                                       "reference native entry points (oracle/ref_driver.py)", F, E2E_REPEATS)},
                        cpu_baseline={"value": value, "unit": "rays/s", "cores": 1, "kind": "reference",
                                      "sample": "reference CUDA extension (oracle/_ref, unmodified sources compiled for "
                                                "sm_100) on the same B200: the reference has no CPU implementation of "
                                                "this path; %d steps, max_num_locs_per_sample=%d as train.py:136"
                                                % (steps, MAX_LOCS)})
            if not args.no_train:
                line["train"] = train_leg("reference", dev, rank, world, local, steps=4, warmup=2)
        else:
            if rank != 0:
                return
            c = cpu_raycast_baseline()
            line = dict(base, impl="reference", value=c["value"], steps=1, ms_per_step=None, n_gpus=1,
                        clocks={"sm_mhz": None, "sm_max_mhz": None, "reasons": ["cpu run"]}, gpu_launches=0,
                        e2e={"value": c["value"], "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                        cpu_baseline=c)
        if rank == 0:
            print(json.dumps(line))
        if world > 1:
            dist.destroy_process_group()
        return

    o = Ours(dev, rank, B, F, num_sets)
    sampler = ClockSampler(dev.index)
    sampler.start()
    steps = args.steps
    ms, graphs = measure_resident(o.step_fused, num_sets, dev, world, steps, args.warmup)
    sampler.stop_flag = True
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, o.last_outputs(steps))
    del graphs
    value = world * o.rays * steps / (ms * 1e-3)
    ms_e2e, last_loss, copy_only = o.e2e(world, steps, min(args.warmup, 5))
    e2e = world * o.rays * steps / (ms_e2e * 1e-3)
    roof = o.roofline(steps, fused=True) if rank == 0 else None
    extra = {}

    def secondary(name, fn):
        """Secondary legs must not void the headline: on one GPU a failure is recorded in the line instead of raised (with
        several ranks it propagates -- swallowing it on one rank would leave the others waiting in a collective)."""
        try:
            extra[name] = fn()
        except Exception as e:  # noqa: BLE001
            if world > 1:
                raise
            extra[name] = {"error": "%s: %s" % (type(e).__name__, str(e)[:300])}

    def leg_flow():
        n_f = args.steps
        ms_f, loss_f, h2d_f = o.e2e_device_flow(world, n_f, 3)
        return {"value": world * o.rays * n_f / (ms_f * 1e-3), "unit": "rays/s", "ms_per_step": ms_f / n_f, "steps": n_f,
                "h2d_bytes_per_step": h2d_f, "d2h_bytes_per_step": 4, "last_loss": loss_f,
                "api": "dense generator heads resident in HBM -> spsg_b200.sparsify.sparsify_predictions -> normals."
                       "compute_normals_sparse -> losses.render_with_2d_losses -> backward to dense head gradients; only the "
                       "step's frames (depth, colour, labels, cameras) are copied from pinned host memory"}

    def leg_unfused():
        ms_u, _ = measure_resident(o.step_unfused, num_sets, dev, world, steps, 3)
        return {"value": world * o.rays * steps / (ms_u * 1e-3), "unit": "rays/s", "ms_per_step": ms_u / steps,
                "steps": steps, "note": "same workload at the reference op boundary: forward renders, backward takes four "
                                          "upstream gradient images (no fused losses)"}

    def leg_c2():
        sets2, _ = auto_sets(1, 1)
        o2 = Ours(dev, rank, 1, 1, sets2)
        ms2, _ = measure_resident(o2.step_fused, sets2, dev, world, steps, 3)
        return {"workload": "c2: one chunk x one 320x256 view (BASELINE configs[1]), fused losses", "unit": "rays/s",
                "value": world * o2.rays * steps / (ms2 * 1e-3), "ms_per_step": ms2 / steps, "steps": steps}

    if not args.no_secondary:
        secondary("e2e_train_flow", leg_flow)
        secondary("unfused", leg_unfused)
        if args.workload != "c2":
            secondary("c2", leg_c2)
    # per step: fill, index, cell classes, forward (its last CTA finalises the loss), gather
    launches = 5
    if not args.no_train:
        o.mods, o.devsets, o.returned = None, None, None
        torch.cuda.empty_cache()
        def leg_train():
            # the step as this package runs it on B200 (generator in NDHWC), and the same step with the generator left in
            # PyTorch's default layout -- the reference arm's configuration -- so that the layout's share is visible
            t = train_leg("ours", dev, rank, world, local, layout="ndhwc")
            torch.cuda.empty_cache()
            d = train_leg("ours", dev, rank, world, local, steps=4, warmup=2, layout="ncdhw")
            t["default_layout"] = {k: d[k] for k in ("chunks_per_s", "ms_per_step", "steps", "generator_layout", "last_loss") if k in d}
            return t
        secondary("train", leg_train)
    if rank == 0:
        line = dict(base, value=value, steps=steps, ms_per_step=ms / steps, clocks=sampler.summary(),
                    e2e={"value": e2e, "unit": "rays/s", "h2d_bytes_per_step": copy_only.pop("h2d_bytes_per_step"),
                         "host_input_bytes_per_step": bytes_of(o.host[0], H2D_KEYS),
                         "d2h_bytes_per_step": 4, "steps": steps, "ms_per_step": ms_e2e / steps,
                         "api": "host inputs in the reference's formats -> spsg_b200.raycast_rgbd_cuda.pack_locs_host (int64 "
                                "voxel rows -> uint32 cell indices, %d host threads, every step) -> one pinned staging buffer "
                                "copied on a copy stream (double-buffered) -> spsg_b200.losses.render_with_2d_losses (fused "
                                "raycast + depth/colour/semantic losses) + backward; median of %d timed regions"
                                % (copy_only.pop("host_pack_threads"), E2E_REPEATS),
                         "last_loss": last_loss,
                         "h2d_copy_only": dict(copy_only, note="the step's pinned host -> device copy alone, all ranks at once: "
                                                               "the floor of this leg on this host")},
                    gpu_launches=launches * steps, roofline=roof, **extra)
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_raycast_baseline()
            try:
                line["cpu_baseline"]["generator_config1"] = cpu_generator_baseline()
            except Exception as e:  # noqa: BLE001
                line["cpu_baseline"]["generator_config1"] = {"error": "%s: %s" % (type(e).__name__, str(e)[:300])}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
