"""Whole-room inference by sliding chunks, with multi-view semantic rendering of every chunk, sharded over GPUs
(BASELINE.json configs[4]; SURVEY.md section 8(f) rank 2).

The reference's ``test_scene_as_chunks.py`` slides a (Dz, 64, 64) window with stride 32 over the room
(test_scene_as_chunks.py:156-157), runs the generator on every window and blends the overlapping outputs; it renders
nothing.  This driver adds the rendering: every window's predicted sparse voxels are ray-cast from ``views_per_chunk``
cameras around the window (camera set-up as in test_scene.py:89-95: fixed intrinsics, camera->grid pose per view) with the
B200 raycaster, several windows per launch.  Windows are independent, so ranks take them round-robin
(``parallel.shard_round_robin``) and nothing is exchanged on the data path; per-class pixel counts are summed over ranks
at the end (one tiny all-reduce).

The generator itself is out of scope (stock PyTorch, SURVEY.md section 2): ``predict`` is any callable that maps a window
to its predicted sparse voxels; ``synthetic_predictor`` stands in for it with the analytic room of ``synthetic.py``.
"""
import math

import numpy as np
import torch

from . import parallel as P
from . import synthetic as S
from .losses import labels_from_render
from .raycast_rgbd import RaycastRGBD


def chunk_windows(room_dims_zyx, chunk_yx=(64, 64), stride=32):
    """(y0, x0) of every window, in the reference's enumeration order (test_scene_as_chunks.py:156-157)."""
    return [(y, x) for y in range(0, room_dims_zyx[1], stride) for x in range(0, room_dims_zyx[2], stride)]


def window_views(num_views, chunk_dims_zyx, radius=75.0, height=70.0):
    """camera->grid matrices (num_views,4,4) around one chunk (grid = the chunk's own voxel frame) and intrinsics."""
    cz, cy, cx = chunk_dims_zyx[0] * 0.3125, chunk_dims_zyx[1] * 0.5, chunk_dims_zyx[2] * 0.5
    mats = []
    for k in range(num_views):
        az = math.radians(360.0 * k / num_views + 5.0)
        eye = (cx + radius * math.cos(az), cy + radius * math.sin(az), height)
        mats.append(S.look_at(eye, (cx, cy, cz)))
    view = np.stack(mats).astype(np.float32)
    intr = np.tile(np.asarray(S.INTRINSICS, dtype=np.float32), (num_views, 1))
    return view, intr


def _payload_from_positions(gz, gy, gx, seed):
    """Deterministic stand-in payload of a voxel from its room coordinates (so that it does not depend on how windows are
    grouped into launches or dealt to ranks): colour in [0,1)^3 and 14 logits with standard deviation 14."""
    key = (gz * 73856093) ^ (gy * 19349663) ^ (gx * 83492791) ^ (seed * 2654435761)
    salts = torch.arange(1, 4 + S.NUM_CLASSES, device=key.device, dtype=torch.int64) * 0x9E3779B97F4A7C1
    h = key[:, None] * 6364136223846793005 + salts[None, :]          # int64 arithmetic wraps
    h = (h ^ (h >> 29)) * 0x3F58476D1CE4E5B9
    h = h ^ (h >> 32)
    u = ((h >> 11) & 0xFFFFFF).to(torch.float32) / 16777216.0
    return u[:, :3].contiguous(), ((u[:, 3:] - 0.5) * 48.5).contiguous()


def synthetic_predictor(room_sdf, truncation=S.TRUNCATION, seed=0):
    """Stand-in for generator + sparsification (train.py:494-509) on a dense room SDF tensor (Dz,Dy,Dx) that lives on the
    GPU.  The "generator heads" are dense room volumes made once: the SDF itself, a colour volume (3 channels) and a
    logit volume (14 channels), both a fixed function of the voxel's room coordinates (so a window's payload does not
    depend on launch grouping or rank).  Returns ``predict(y0, x0, chunk_yx) -> (locs (n,3) int64 z,y,x in chunk
    coordinates, sdf (n,1), colour (n,3), semantic logits (n,14))``; ``predict.predict_group(windows, chunk_yx) -> (locs
    (n,4) with b = index into windows, sdf, colour, logits)`` does a whole launch group at once: the windows' heads are
    stacked as dense (B,C,Dz,cy,cx) batches, like a generator's output, and go through ``sparsify.sparsify_predictions``
    (one host synchronisation per group)."""
    from . import sparsify
    dz, dy, dx = room_sdf.shape
    dev = room_sdf.device
    gz, gy, gx = torch.meshgrid(torch.arange(dz, device=dev), torch.arange(dy, device=dev), torch.arange(dx, device=dev),
                                indexing="ij")
    color, sem = _payload_from_positions(gz.reshape(-1), gy.reshape(-1), gx.reshape(-1), seed)
    room_color = color.t().reshape(3, dz, dy, dx).contiguous()
    room_sem = sem.t().reshape(S.NUM_CLASSES, dz, dy, dx).contiguous()
    del gz, gy, gx, color, sem
    outside = 2.0 * truncation + 1.0

    def predict(y0, x0, chunk_yx):
        win = room_sdf[:, y0:y0 + chunk_yx[0], x0:x0 + chunk_yx[1]]
        locs = torch.nonzero(win.abs() < truncation)
        z, y, x = locs[:, 0], locs[:, 1] + y0, locs[:, 2] + x0
        return (locs, room_sdf[z, y, x].reshape(-1, 1).contiguous(), room_color[:, z, y, x].t().contiguous(),
                room_sem[:, z, y, x].t().contiguous())

    cache = {}

    def assemble(windows, chunk_yx):
        """The dense heads a generator would output for this launch group: (B,1|3|14,Dz,cy,cx)."""
        B = len(windows)
        head_sdf = torch.full((B, 1, dz, chunk_yx[0], chunk_yx[1]), outside, device=dev)
        head_col = torch.zeros(B, 3, dz, chunk_yx[0], chunk_yx[1], device=dev)
        head_sem = torch.zeros(B, S.NUM_CLASSES, dz, chunk_yx[0], chunk_yx[1], device=dev)
        for b, (y0, x0) in enumerate(windows):
            ys, xs = slice(y0, y0 + chunk_yx[0]), slice(x0, x0 + chunk_yx[1])
            win = room_sdf[:, ys, xs]                                           # smaller at the room border
            head_sdf[b, 0, :, :win.shape[1], :win.shape[2]] = win
            head_col[b, :, :, :win.shape[1], :win.shape[2]] = room_color[:, :, ys, xs]
            head_sem[b, :, :, :win.shape[1], :win.shape[2]] = room_sem[:, :, ys, xs]
        return head_sdf, head_col, head_sem

    def prepare_groups(groups, chunk_yx):
        """Assemble (and keep) the heads of these launch groups ahead of time, so that a timed run measures the path from
        the generator's outputs on, not the stand-in's slicing."""
        for g in groups:
            cache[(tuple(g), tuple(chunk_yx))] = assemble(g, chunk_yx)

    def predict_group(windows, chunk_yx):
        heads = cache.get((tuple(windows), tuple(chunk_yx)))
        if heads is None:
            heads = assemble(windows, chunk_yx)
        return sparsify.sparsify_predictions(heads[0], truncation, None, heads[1], heads[2])

    predict.prepare_groups = prepare_groups
    predict.predict_group = predict_group
    return predict


def render_room(predict, room_dims_zyx, device, views_per_chunk=5, chunks_per_launch=8, chunk_yx=(64, 64), stride=32,
                width=S.WIDTH, height=S.HEIGHT, rank=0, world=1, max_num_locs_per_sample=640000, keep_images=False):
    """Render this rank's share of the room's windows.  Returns dict(windows, rendered_windows, rays, label_hist (15,)
    summed over ranks, images: list of (window, labels (F,H,W) uint8) when ``keep_images``)."""
    dz = room_dims_zyx[0]
    chunk_dims = (dz, chunk_yx[0], chunk_yx[1])
    windows = chunk_windows(room_dims_zyx, chunk_yx, stride)
    mine = [windows[i] for i in P.shard_round_robin(len(windows), rank, world)]
    B, F = chunks_per_launch, views_per_chunk
    rc = RaycastRGBD(B, chunk_dims, width, height, S.DEPTH_MIN, S.DEPTH_MAX, S.THRESH_SAMPLE_DIST, S.RAY_INCREMENT,
                     max_num_frames=F, max_num_locs_per_sample=max_num_locs_per_sample, device=device)
    view_np, intr_np = window_views(F, chunk_dims)
    view = torch.from_numpy(np.tile(view_np, (B, 1, 1))).to(device)
    intr = torch.from_numpy(np.tile(intr_np, (B, 1))).to(device)
    hist = torch.zeros(S.NUM_CLASSES + 1, dtype=torch.int64, device=device)
    images, rendered, rays = [], 0, 0
    predict_group = getattr(predict, "predict_group", None)
    for s in range(0, len(mine), B):
        group = mine[s:s + B]
        if predict_group is not None:
            # the whole group at once; chunk slot b = position in the group, windows without voxels keep an idle slot
            locs, sdf, color, sem = predict_group(group, chunk_yx)
            edges = torch.searchsorted(locs[:, 3].contiguous(), torch.arange(len(group) + 1, device=device)).tolist()
            present = [b for b in range(len(group)) if edges[b + 1] > edges[b]]   # rows are sorted by chunk
            slots = len(group)
        else:
            parts = [predict(y0, x0, chunk_yx) for (y0, x0) in group]
            present = [k for k, p in enumerate(parts) if p[0].shape[0] > 0]
            slots = len(present)
            if present:  # non-empty windows packed into consecutive chunk slots
                locs = torch.cat([torch.cat([parts[k][0], torch.full((parts[k][0].shape[0], 1), b, dtype=torch.long,
                                                                     device=device)], 1)
                                  for b, k in enumerate(present)]).contiguous()
                sdf = torch.cat([parts[k][1] for k in present])
                color = torch.cat([parts[k][2] for k in present])
                sem = torch.cat([parts[k][3] for k in present])
        if not present:  # the reference skips empty windows (test_scene_as_chunks.py:160-161)
            continue
        with torch.no_grad():
            # pred2d_label of train.py:749-752 and its per-class pixel counts.  A pixel's rendered logits are its hit
            # voxel's row, so its label is the label of that row: one byte per voxel, then the label render (which writes
            # no float image and needs no normals or colours)
            voxel_labels = labels_from_render(sem)
            labels, h = rc.render_labels(locs, sdf, voxel_labels, view, intr, histogram=True)
            labels = labels[:slots * F].view(slots, F, height, width)
            # idle slots, and the slots past this group's windows, rendered nothing: all their pixels are label 14
            h[S.NUM_CLASSES] -= (B - len(present)) * F * width * height
            if len(present) < slots:
                labels = labels[torch.tensor(present, device=device)]
            hist += h
        rendered += len(present)
        rays += len(present) * F * width * height
        if keep_images:
            for j, k in enumerate(present):
                images.append((group[k], labels[j].cpu()))
    total_hist = hist.clone()
    if world > 1 and torch.distributed.is_available() and torch.distributed.is_initialized():
        torch.distributed.all_reduce(total_hist)   # the only collective: 15 counters
    return dict(windows=len(windows), rendered_windows=rendered, rays=rays,
                label_hist=total_hist.cpu().numpy().astype(np.float64),
                images=images)


def labels_from_render_logits(sem_img, depth):
    """Per-pixel predicted class of a rendering of semantic *logits* (train.py:749-752: argmax over the 14 logits),
    14 where the ray hit nothing."""
    lab = sem_img.argmax(dim=-1)
    return torch.where(depth != -float("inf"), lab, torch.full_like(lab, S.NUM_CLASSES)).to(torch.uint8)


def synthetic_room_sdf(room_dims_zyx, device, seed=0):
    """Analytic room: the chunk scene of ``synthetic.sdf_volume`` repeated with period 64 in y and x plus the outer floor,
    as one dense float32 tensor (Dz,Dy,Dx) on ``device``."""
    dz, dy, dx = room_dims_zyx
    base, _ = S.sdf_volume(seed, (dz, 64, 64))
    reps = (1, (dy + 63) // 64, (dx + 63) // 64)
    room = np.tile(base, reps)[:, :dy, :dx]
    return torch.from_numpy(np.ascontiguousarray(room)).to(device)
