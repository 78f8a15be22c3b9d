"""2D view-guided losses fused into the raycast (SURVEY.md section 8 rows a11-a13).

``render_with_2d_losses`` renders the predicted chunk exactly like ``RaycastRGBD.forward`` and, in the same
kernel, accumulates the reference's three 2D loss terms

    depth L1      mean |depth * voxelsize - images_depth|  over (hit & images_depth != 0)    train.py:635-638
    colour L1     mean |colour * w - target * w|            over hit pixels x 3 channels      loss.py:246-257
    semantic CE   sum w[y] * nll / sum w[y]                 over (hit & label < 14)           train.py:744-746

Its backward never materialises the loss terms' gradient images: every registered pixel's gradient is recomputed from
(rendering, target, normalisers) inside the per-voxel gather, which can also add the caller's own gradient images of the
renderings (``differentiable_images=True``).  No CPU path.
"""
import ctypes

import torch
from torch.autograd import Function

from . import _native as N
from . import raycast_rgbd_cuda as rc


def labels_from_render(raycast_semantic, histogram=False):
    """target2d_label of train.py:614-616 / pred2d_label of :749-752: ``argmax(cat(render, ones), -1)`` as uint8
    (14 = miss or unlabeled), shape ``raycast_semantic.shape[:-1]``, in one pass over the rendering.  With
    ``histogram=True`` also returns the number of pixels per label (15 int64, on the device) from the same pass."""
    sem = raycast_semantic.detach()
    rc._check_input(sem, "raycast_semantic")
    rc._check_dtype(sem, torch.float32, "raycast_semantic")
    if sem.shape[-1] != 14:
        raise RuntimeError("raycast_semantic must have 14 channels")
    if sem.data_ptr() % 8:
        sem = sem.clone()
    labels = torch.empty(sem.shape[:-1], dtype=torch.uint8, device=sem.device)
    hist = torch.empty(15, dtype=torch.int64, device=sem.device) if histogram else None
    with rc.device_guard(sem.device):
        N.check(N.lib.spsg_labels_from_render(N.ptr(sem), labels.numel(), N.ptr(labels), N.ptr(hist),
                                              rc._stream(sem.device)))
    return (labels, hist) if histogram else labels


def _targets_struct(images, h, w, target_depth, target_color, weight_color, target_label, class_weight, voxelsize,
                    weights):
    def chk(t, numel, dtype, name):
        if t is None:
            return None
        if not t.is_cuda or not t.is_contiguous() or t.dtype != dtype or t.numel() != numel:
            raise RuntimeError("%s must be a contiguous CUDA %s tensor with %d elements" % (name, dtype, numel))
        return t
    px = images * h * w
    t = N.LossTargets(N.ptr(chk(target_depth, px, torch.float32, "target_depth")),
                      N.ptr(chk(target_color, 3 * px, torch.float32, "target_color")),
                      N.ptr(chk(weight_color, px, torch.float32, "weight_color")),
                      N.ptr(chk(target_label, px, torch.uint8, "target_label")),
                      N.ptr(chk(class_weight, 14, torch.float32, "class_weight")),
                      float(voxelsize), float(weights[0]), float(weights[1]), float(weights[2]))
    return t


def _module_workspace(m):
    ws = getattr(m, "workspace", None)
    if ws is None:  # a raycaster-like object without one: give it one
        ws = m.workspace = rc.ModuleWorkspace()
    return ws


def fused_forward(m, locs, vals_sdf, vals_colors, vals_normals, vals_semantic, view_matrix, intrinsic_params, targets,
                  clear_grads):
    """``spsg_raycast_forward_loss`` on the buffers of raycaster ``m``: validates every tensor whose pointer crosses the
    C ABI, renders, accumulates the 2D loss terms.  ``targets`` = (target_depth, target_color, weight_color, target_label,
    class_weight, voxelsize, (w_depth, w_colour, w_semantic)).  ``vals_normals`` (N,3) shared or (N,F,3) per view
    (SPSG_FLAG_VIEW_NORMALS, set in the returned params).  Returns (params, targets struct, loss_out[8])."""
    images = view_matrix.shape[0]
    views = max(1, images // m.batch_size)
    if images != views * m.batch_size or views > m.max_num_frames:
        raise RuntimeError("view_matrix has %d images: expected batch_size (%d) x views <= max_num_frames (%d)"
                           % (images, m.batch_size, m.max_num_frames))
    per_view = rc.view_normals(vals_normals, views)
    n = rc.check_voxel_inputs(locs, vals_sdf, vals_colors, vals_normals, vals_semantic, view_matrix, intrinsic_params,
                              images, views if per_view else 1)
    if n * views > m.mapping3dto2d.shape[0]:
        raise RuntimeError("too many voxels for raycast (%d x %d views > %d rows)" % (n, views, m.mapping3dto2d.shape[0]))
    d_normal = rc.normal_grad_buffer(m, per_view)
    if clear_grads and (m.d_depth.shape[0] < n or m.d_color.shape[0] < n or
                        d_normal.shape[0] < n * (views if per_view else 1) or m.d_semantic.shape[0] < n):
        raise RuntimeError("d_* buffers hold fewer than N = %d rows" % n)
    dev = vals_sdf.device
    if m.image_depth.device != dev:
        raise RuntimeError("raycaster buffers live on %s, inputs on %s" % (m.image_depth.device, dev))
    p = N.make_params(m.width, m.height, m.depth_min, m.depth_max, m.thresh_sample_dist, m.ray_increment,
                      m.dims3d[2], m.dims3d[1], m.dims3d[0], m.batch_size, views, m.mapping3dto2d.shape[1], n,
                      rc.with_torch_mode(m.flags | (N.SPSG_FLAG_VIEW_NORMALS if per_view else 0)))
    if rc.is_packed_locs(locs):
        p.flags |= N.SPSG_FLAG_PACKED_LOCS
    target_depth, target_color, weight_color, target_label, class_weight, voxelsize, weights = targets
    tg = _targets_struct(images, m.height, m.width, target_depth, target_color, weight_color, target_label, class_weight,
                         voxelsize, weights)
    # terms, total and normalisers of THIS call (the backward reads the normalisers back)
    loss_out = torch.empty(N.SPSG_LOSS_OUT_FLOATS, device=dev)
    gb = N.grad_buffers(m.d_color, m.d_depth, d_normal, m.d_semantic) if clear_grads else None
    owner = _module_workspace(m)
    with rc.device_guard(dev):
        nbytes = N.workspace_bytes(p)
        prebuilt = owner.take_prebuilt(locs, nbytes)  # index + brick written with locs by sparsify_predictions(raycaster=m)
        ws = owner.get(dev, nbytes)
        p.flags |= prebuilt
        N.check(N.lib.spsg_raycast_forward_loss(
            ctypes.byref(p), N.ptr(m.sparse_mapping), N.ptr(locs), N.ptr(vals_sdf), N.ptr(vals_colors),
            N.ptr(vals_normals), N.ptr(vals_semantic), N.ptr(view_matrix), N.ptr(intrinsic_params),
            N.ptr(m.image_color), N.ptr(m.image_depth), N.ptr(m.image_normal), N.ptr(m.image_semantic),
            N.ptr(m.mapping3dto2d), N.ptr(m.mapping3dto2d_num), ctypes.byref(tg), N.ptr(loss_out),
            ctypes.byref(gb) if gb is not None else None, N.ptr(ws), ws.numel(), rc._stream(dev)))
        owner.filled(p)
        if prebuilt:
            owner.mark_prebuilt(locs)
            p.flags &= ~N.SPSG_FLAG_INDEX_PREBUILT  # (the params go on to the backward)
        p.flags &= ~N.SPSG_FLAG_PACKED_LOCS
    return p, tg, loss_out


def _upstream_struct(m, p, upstream):
    """``spsg_upstream_grads`` of ``upstream`` = (grad_color, grad_depth, grad_normal, grad_semantic), any of them None:
    contiguous float32 CUDA tensors shaped like the renderings of the forward ``p`` describes."""
    images = p.num_chunks * p.views_per_chunk
    px = images * p.height * p.width
    ptrs = []
    for g, ch, name in zip(upstream, (3, 1, 3, 14), ("grad_color", "grad_depth", "grad_normal", "grad_semantic")):
        if g is not None:
            rc._check_input(g, name)
            rc._check_dtype(g, torch.float32, name)
            if g.numel() != ch * px or g.device != m.image_depth.device:
                raise RuntimeError("%s must hold %d x %d x %d x %d floats on %s" % (name, images, p.height, p.width, ch,
                                                                                   m.image_depth.device))
        ptrs.append(N.ptr(g))
    return N.UpstreamGrads(*ptrs)


def _per_view(p):
    return bool(p.flags & N.SPSG_FLAG_VIEW_NORMALS)


def _voxel_grads(m, p, n):
    """(d_sdf, d_color, d_normal, d_semantic): rows [0, N) of ``m.d_*``; per-view normals as (N,F,3)."""
    d_normal = rc.normal_grad_buffer(m, _per_view(p))
    d_normal = d_normal[:n * p.views_per_chunk].view(n, p.views_per_chunk, 3) if _per_view(p) else d_normal[:n]
    return m.d_depth[:n], m.d_color[:n], d_normal, m.d_semantic[:n]


def fused_backward(m, p, tg, loss_out, grad_scale, grads_cleared, upstream=None):
    """``spsg_raycast_backward_loss``: voxel gradients of ``grad_scale * total`` into rows [0, N) of ``m.d_*`` (the
    per-view normal rows of ``raycast_rgbd_cuda.normal_grad_buffer`` when ``p`` has SPSG_FLAG_VIEW_NORMALS).
    ``upstream`` = (grad_color, grad_depth, grad_normal, grad_semantic) gradient images of the renderings (any of them
    None; contiguous float32): ``spsg_raycast_backward_loss_upstream`` then adds them, unscaled, in the same gather.
    ``grad_scale`` None means 1.  Runs in the deterministic mode of this call (``m.flags`` or torch's switch): the
    workspace check refuses a forward that ran in the other."""
    det = rc.with_torch_mode(m.flags) & N.SPSG_FLAG_DETERMINISTIC
    if grads_cleared or (p.flags & N.SPSG_FLAG_DETERMINISTIC) != det:
        p = type(p).from_buffer_copy(p)  # the caller's params stay as the forward left them
        p.flags = (p.flags & ~N.SPSG_FLAG_DETERMINISTIC) | det
        if grads_cleared:
            p.flags |= N.SPSG_FLAG_GRADS_CLEARED
    dev = m.image_depth.device
    if grad_scale is not None:
        rc._check_input(grad_scale, "grad_scale")
        rc._check_dtype(grad_scale, torch.float32, "grad_scale")
    up = _upstream_struct(m, p, upstream) if upstream is not None else None
    d_normal = rc.normal_grad_buffer(m, _per_view(p))
    owner = _module_workspace(m)
    with rc.device_guard(dev):
        ws = owner.check(p, N.workspace_bytes(p))  # the work list of the forward that rendered m's images
        if up is None:
            N.check(N.lib.spsg_raycast_backward_loss(
                ctypes.byref(p), N.ptr(m.image_color), N.ptr(m.image_depth), N.ptr(m.image_semantic),
                ctypes.byref(tg), N.ptr(loss_out), N.ptr(grad_scale), N.ptr(m.sparse_mapping), N.ptr(m.mapping3dto2d),
                N.ptr(m.mapping3dto2d_num), N.ptr(m.d_color), N.ptr(m.d_depth), N.ptr(d_normal), N.ptr(m.d_semantic),
                N.ptr(ws), ws.numel(), rc._stream(dev)))
        else:
            N.check(N.lib.spsg_raycast_backward_loss_upstream(
                ctypes.byref(p), N.ptr(m.image_color), N.ptr(m.image_depth), N.ptr(m.image_semantic),
                ctypes.byref(tg), N.ptr(loss_out), N.ptr(grad_scale), ctypes.byref(up), N.ptr(m.sparse_mapping),
                N.ptr(m.mapping3dto2d), N.ptr(m.mapping3dto2d_num), N.ptr(m.d_color), N.ptr(m.d_depth),
                N.ptr(d_normal), N.ptr(m.d_semantic), N.ptr(ws), ws.numel(), rc._stream(dev)))


def _targets_off(tg):
    """A copy of the targets struct with every loss term switched off: the fused backward then gathers the upstream
    images alone."""
    return N.LossTargets(None, None, None, None, None, tg.voxelsize, tg.weight_depth, tg.weight_color_loss,
                         tg.weight_semantic)


class FusedRaycastLossFunction(Function):
    @staticmethod
    def forward(ctx, raycaster, locs, vals_sdf, vals_colors, vals_normals, vals_semantic, view_matrix,
                intrinsic_params, target_depth, target_color, weight_color, target_label, class_weight, voxelsize,
                weights, differentiable_images=False):
        m = raycaster
        n = locs.shape[0]
        images = view_matrix.shape[0]
        # gradients that do not reach an output stay None: no zero-filled image per non-differentiable rendering
        ctx.set_materialize_grads(False)
        # a backward will follow: let the forward's fill pass clear the gradient rows it will write
        ctx.grads_cleared = any(ctx.needs_input_grad[2:6]) and n > 0
        p, tg, loss_out = fused_forward(m, locs, vals_sdf, vals_colors, vals_normals, vals_semantic, view_matrix,
                                        intrinsic_params, (target_depth, target_color, weight_color, target_label,
                                                           class_weight, voxelsize, weights), ctx.grads_cleared)
        ctx.raycaster, ctx.params, ctx.targets, ctx.n, ctx.loss_out = m, p, tg, n, loss_out
        ctx.forward_id = m.workspace.forwards
        # keep the target tensors alive until backward (the struct only holds raw pointers)
        ctx.keep = (target_depth, target_color, weight_color, target_label, class_weight)
        ctx.differentiable_images = differentiable_images
        imgs = (m.image_color, m.image_depth, m.image_normal, m.image_semantic)
        if not differentiable_images:
            ctx.mark_non_differentiable(*imgs)
        if images != m.image_depth.shape[0] or differentiable_images:
            # differentiable: always views, so that the module's buffers themselves never carry this node's history
            # (the next forward of the module takes them as inputs, and must not link its graph to this one)
            imgs = tuple(i[:images] for i in imgs)
            if not differentiable_images:
                ctx.mark_non_differentiable(*imgs)
        if differentiable_images:
            # the backward recomputes the loss gradients from these buffers: saving them makes an in-place change
            # before backward() an error (autograd's version counter) instead of silently wrong gradients
            ctx.save_for_backward(*imgs)
        terms = loss_out[:3]
        ctx.mark_non_differentiable(terms)
        return (loss_out[3], terms) + imgs

    @staticmethod
    def backward(ctx, grad_total, grad_terms, *grad_images):
        m, n = ctx.raycaster, ctx.n
        upstream = None
        if ctx.differentiable_images:
            ctx.saved_tensors  # noqa: B018 -- raises if a rendering was modified in place since the forward
            if any(g is not None for g in grad_images):
                upstream = tuple(None if g is None else g.to(torch.float32).contiguous() for g in grad_images)
        if grad_total is None and upstream is None:
            return (None,) * 16
        m.workspace.check_latest(ctx.forward_id)
        if grad_total is None:
            # only the images feed the objective: no scale derived from the loss normalisers (an empty valid set would
            # turn 0 * (w / 0) into NaN); the targets switched off leave the plain gather of the upstream images
            fused_backward(m, ctx.params, _targets_off(ctx.targets), ctx.loss_out, None, ctx.grads_cleared, upstream)
        else:
            fused_backward(m, ctx.params, ctx.targets, ctx.loss_out, grad_total.to(torch.float32).contiguous(),
                           ctx.grads_cleared, upstream)
        ctx.grads_cleared = False  # the forward cleared the rows once: a second backward (retain_graph) clears its own
        grads = _voxel_grads(m, ctx.params, n)
        m.workspace.grad_views = grads  # leaves get copies, not the buffers (raycast_rgbd_cuda.ModuleWorkspace)
        return (None, None) + grads + (None,) * 10


def render_loss_and_voxel_grads(raycaster, locs, vals_sdf, vals_colors, vals_normals, vals_semantics, view_matrix,
                                intrinsic_params, images_depth=None, images_color=None, weight_color=None,
                                target2d_label=None, weight_semantic_class=None, voxelsize=0.02, weight_depth_loss=1.0,
                                weight_color_loss=1.0, weight_semantic_loss=1.0, grad_scale=None):
    """The fused forward + backward pair without autograd, for callers that own the voxel tensors' gradients themselves
    (and for CUDA-graph capture: nothing but the two native calls is enqueued).  Returns ``(loss_out, (d_sdf, d_color,
    d_normal, d_semantic))``: ``loss_out[0:3]`` = depth / colour / semantic terms, ``loss_out[3]`` = weighted total; the
    gradients of ``grad_scale * total`` (default 1) are views of rows [0, N) of the raycaster's ``d_*`` buffers; with
    per-view normals ``(N,F,3)`` the normal gradient is ``(N,F,3)`` too."""
    c = lambda t: None if t is None else t.contiguous()
    m, n = raycaster, locs.shape[0]
    p, tg, loss_out = fused_forward(m, locs, vals_sdf, vals_colors, vals_normals, vals_semantics, view_matrix,
                                    intrinsic_params, (c(images_depth), c(images_color), c(weight_color), c(target2d_label),
                                                       weight_semantic_class, voxelsize,
                                                       (weight_depth_loss, weight_color_loss, weight_semantic_loss)), n > 0)
    if grad_scale is None:
        grad_scale = getattr(m, "_unit_scale", None)
        if grad_scale is None or grad_scale.device != loss_out.device:
            grad_scale = m._unit_scale = torch.ones((), device=loss_out.device)
    fused_backward(m, p, tg, loss_out, grad_scale, n > 0)
    return loss_out, _voxel_grads(m, p, n)


def render_with_2d_losses(raycaster, locs, vals_sdf, vals_colors, vals_normals, vals_semantics, view_matrix,
                          intrinsic_params, images_depth=None, images_color=None, weight_color=None,
                          target2d_label=None, weight_semantic_class=None, voxelsize=0.02,
                          weight_depth_loss=1.0, weight_color_loss=1.0, weight_semantic_loss=1.0,
                          differentiable_images=False):
    """Fused prediction raycast + 2D losses (train.py:626-643, 744-746 in one kernel pair).

    raycaster        a ``RaycastRGBD`` (owns the image / mapping / gradient buffers, as in the reference)
    images_depth     (I,H,W) or (I,1,H,W) metres, 0 = hole;  None switches the depth term off
    images_color     (I,H,W,3) channels-last (the reference passes images_color.permute(0,2,3,1)); None = off
    weight_color     (I,H,W) or (I,1,H,W) per-pixel colour weight or None
    target2d_label   (I,H,W) or (I,H,W,1) uint8, 14 = ignore; None switches the semantic term off
    Returns (total, terms[3] = (depth, colour, semantic), (color, depth, normal, semantic) renderings).
    ``total = weight_depth_loss*depth + weight_color_loss*colour + weight_semantic_loss*semantic``; ``terms`` are
    reported values, like the ``.item()`` logging in train.py.  Gradients flow from ``total`` and, with
    ``differentiable_images=True``, from the four renderings too: terms the caller computes on them (a discriminator on
    ``cat(colour, normal)``, a style loss) are gathered into the voxels by the same backward launch, per registered pixel.

    The renderings are the raycaster's own buffers, as in the reference: any later forward of the same module overwrites
    them, so this must be the last call on ``raycaster`` before ``backward()`` (clone what is needed beyond that).  With
    ``differentiable_images=True`` they are saved for the backward, and modifying one in place before ``backward()``
    raises autograd's version-counter error."""
    if vals_semantics is None:
        vals_semantics = torch.zeros(vals_sdf.shape[0], 14, device=vals_sdf.device)
    out = FusedRaycastLossFunction.apply(
        raycaster, locs, vals_sdf, vals_colors, vals_normals, vals_semantics, view_matrix, intrinsic_params,
        None if images_depth is None else images_depth.contiguous(),
        None if images_color is None else images_color.contiguous(),
        None if weight_color is None else weight_color.contiguous(),
        None if target2d_label is None else target2d_label.contiguous(),
        weight_semantic_class, voxelsize, (weight_depth_loss, weight_color_loss, weight_semantic_loss),
        bool(differentiable_images))
    return out[0], out[1], out[2:]


# ---------------------------------------------------------------------------------------------------------------------
# The same three terms as stand-alone ops on rendered images: the boundary at which the reference applies them
# (loss.compute_2dcolor_loss, loss.py:246-257; the inline expressions of train.py:635-638 and :744-746).  One pass over
# the pixels instead of a boolean-mask select (which synchronises the host) + several element-wise kernels.
# ---------------------------------------------------------------------------------------------------------------------

class _Losses2D(Function):
    @staticmethod
    def forward(ctx, image_color, image_depth, image_semantic, target_depth, target_color, weight_color, target_label,
                class_weight, voxelsize, weights):
        some = next(t for t in (image_color, image_depth, image_semantic) if t is not None)
        dev = some.device
        px = {"c": None if image_color is None else image_color.numel() // 3,
              "d": None if image_depth is None else image_depth.numel(),
              "s": None if image_semantic is None else image_semantic.numel() // 14}
        num_pixels = next(v for v in px.values() if v is not None)
        if any(v is not None and v != num_pixels for v in px.values()):
            raise RuntimeError("renderings disagree on the number of pixels")
        for t, name in ((image_color, "image_color"), (image_depth, "image_depth"), (image_semantic, "image_semantic")):
            if t is not None:
                rc._check_input(t, name)
                rc._check_dtype(t, torch.float32, name)
        tg = _targets_struct(1, 1, num_pixels, target_depth, target_color, weight_color, target_label, class_weight,
                             voxelsize, weights)
        loss_out = torch.empty(N.SPSG_LOSS_OUT_FLOATS, device=dev)
        # deterministic algorithms: the sums in pixel order (per-block partials in a scratch that grows with the image)
        det = torch.are_deterministic_algorithms_enabled()
        forward = N.lib.spsg_losses2d_forward_deterministic if det else N.lib.spsg_losses2d_forward
        scratch = torch.empty(N.lib.spsg_losses2d_deterministic_scratch_bytes(num_pixels) if det else 4096,
                              dtype=torch.uint8, device=dev)
        with rc.device_guard(dev):
            N.check(forward(ctypes.byref(tg), N.ptr(image_color), N.ptr(image_depth), N.ptr(image_semantic), num_pixels,
                            N.ptr(loss_out), N.ptr(scratch), scratch.numel(), rc._stream(dev)))
        ctx.targets, ctx.num_pixels, ctx.loss_out = tg, num_pixels, loss_out
        ctx.keep = (target_depth, target_color, weight_color, target_label, class_weight)
        ctx.save_for_backward(*[t for t in (image_color, image_depth, image_semantic) if t is not None])
        ctx.present = tuple(t is not None for t in (image_color, image_depth, image_semantic))
        terms = loss_out[:3]
        ctx.mark_non_differentiable(terms)
        return loss_out[3], terms

    @staticmethod
    def backward(ctx, grad_total, grad_terms):
        saved = list(ctx.saved_tensors)
        imgs = [saved.pop(0) if p else None for p in ctx.present]
        dev = ctx.loss_out.device
        need = ctx.needs_input_grad[:3]
        grads = [torch.empty_like(t) if (t is not None and n) else None for t, n in zip(imgs, need)]
        scale = grad_total.to(torch.float32).contiguous()
        with rc.device_guard(dev):
            N.check(N.lib.spsg_losses2d_backward(ctypes.byref(ctx.targets), N.ptr(imgs[0]), N.ptr(imgs[1]), N.ptr(imgs[2]),
                                                 ctx.num_pixels, N.ptr(ctx.loss_out), N.ptr(scale), N.ptr(grads[0]),
                                                 N.ptr(grads[1]), N.ptr(grads[2]), rc._stream(dev)))
        return (grads[0], grads[1], grads[2]) + (None,) * 7


def losses_2d(raycast_color=None, raycast_depth=None, raycast_semantic=None, images_depth=None, images_color=None,
              weight_color=None, target2d_label=None, weight_semantic_class=None, voxelsize=0.02,
              weight_depth_loss=1.0, weight_color_loss=1.0, weight_semantic_loss=1.0):
    """All requested 2D terms of rendered images in one pass.  Returns (total, terms[3] = depth, colour, semantic);
    gradients flow from ``total`` into the renderings."""
    c = lambda t: None if t is None else t.contiguous()
    return _Losses2D.apply(c(raycast_color) if images_color is not None else None,
                           c(raycast_depth) if images_depth is not None else None,
                           c(raycast_semantic) if target2d_label is not None else None,
                           c(images_depth), c(images_color), c(weight_color), c(target2d_label), weight_semantic_class,
                           voxelsize, (weight_depth_loss, weight_color_loss, weight_semantic_loss))


def depth_l1_loss(raycast_depth, images_depth, voxelsize):
    """train.py:635-638: mean |raycast_depth * voxelsize - images_depth| over (rendered & images_depth != 0)."""
    return losses_2d(raycast_depth=raycast_depth, images_depth=images_depth, voxelsize=voxelsize)[0]


def color_l1_loss(raycast_color, target_color, weight_color=None):
    """Drop-in for loss.compute_2dcolor_loss (loss.py:246-257); ``weight_color`` (B,1,H,W) or None."""
    return losses_2d(raycast_color=raycast_color, images_color=target_color, weight_color=weight_color)[0]


def semantic_2d_ce_loss(raycast_semantic, target2d_label, weight_semantic_class=None):
    """train.py:744-746: class-weighted cross-entropy over (label < 14 & rendered)."""
    return losses_2d(raycast_semantic=raycast_semantic, target2d_label=target2d_label,
                     weight_semantic_class=weight_semantic_class)[0]
