"""Drop-in for the reference's ``torch/utils/raycast_rgbd/raycast_rgbd.py``.

Same classes, constructor arguments, call signatures, buffer attributes and return conventions
(``RayCastRGBDFunction`` raycast_rgbd.py:10-43, ``RaycastRGBD`` :46-85, ``RaycastOcc`` :88-104), so the
reference's ``train.py`` / ``test_scene.py`` run unchanged -- but every native call goes through the C ABI
of ``include/spsg_raycast.h`` (hand-written sm_100a kernels).  There is no CPU path.

Differences, all behind defaulted extras or unobservable through the reference API:
  * several views per chunk: pass ``view_matrix`` / ``intrinsic_params`` with ``B*F`` rows (image ``i`` renders
    chunk ``i // F``, the ordering of reference ``style.compute_view_matrix``, style.py:9-16), ``F <= max_num_frames``.
    The voxel gradient is then the sum over views of the per-view means = F reference calls accumulated by autograd.
  * per-view normals: with ``vals_normals`` of shape ``(N,F,3)``, image ``b*F + f`` renders row ``(v, f)`` -- each view's
    normals in its own camera frame, as F reference calls with their own ``transform`` give (train.py:542-544).  Its
    gradient is ``(N,F,3)``, view f's mean in row ``(v, f)``; ``(N,3)`` keeps the shared payload.
  * no host synchronisation: the reference reads ``locs[-1, -1]`` back to the host (raycast_rgbd.py:22,30).
  * the upstream ``RaycastOcc.forward`` NameError (``raycast_color_cuda``, raycast_rgbd.py:103) is fixed.
  * deterministic mode: under ``torch.use_deterministic_algorithms(True)`` (or with SPSG_FLAG_DETERMINISTIC in ``flags``)
    the voxel -> pixel tables are canonical and the gradients bit-reproducible; forward and backward must agree on it.
  * ``max_pixels_per_voxel=None``: the gradient of a (voxel, view) is the mean over every pixel it received, not over the
    first ``max_pixels_per_voxel`` (SPSG_FLAG_ALL_PIXELS in ``flags``); no ``mapping3dto2d`` table is allocated.
  * ``num_classes=C``: semantic payloads, renderings and gradients of C channels instead of the reference's 14 (1..64;
    e.g. 20 for ScanNet, 41 for NYU40 / mpcat40).  Geometry does not depend on C.
  * ``RaycastRGBD.render_labels``: the label map of a render from one uint8 label per voxel, without the C-wide image.
"""
import torch
from torch import nn
from torch.autograd import Function

from . import _native as N
from . import raycast_rgbd_cuda


class RayCastRGBDFunction(Function):
    @staticmethod
    def forward(ctx, locs, vals_sdf, vals_colors, vals_normals, vals_semantic, view_matrix_inv, intrinsic_params,
                dims3d, width, height, depth_min, depth_max, thresh_sample_dist, ray_increment, image_color,
                image_depth, image_normal, image_semantic, sparse_mapping, mapping3dto2d, mapping3dto2d_num, d_color,
                d_depth, d_normal, d_semantic, views_per_chunk=1, flags=0, workspace_owner=None):
        rows = raycast_rgbd_cuda.table_shape(mapping3dto2d, mapping3dto2d_num, flags)[0]
        if locs.shape[0] * views_per_chunk > rows:  # raycast_rgbd.py:16-21
            print('ERROR: locs size %s vs mapping3dto2d size %s' % (str(locs.shape), str(mapping3dto2d_num.shape if
                  raycast_rgbd_cuda.all_pixels(flags) else mapping3dto2d.shape)))
            keep = rows // views_per_chunk
            locs = locs[:keep]
            vals_sdf = vals_sdf[:keep]
            vals_colors = vals_colors[:keep]
            vals_normals = vals_normals[:keep]
        device = vals_sdf.device
        num_locs = locs.shape[0]
        opts = [width, height, depth_min, depth_max, thresh_sample_dist, ray_increment, dims3d[2], dims3d[1],
                dims3d[0]]  # raycast_rgbd.py:24-25
        # a backward will follow: let the forward's fill pass clear the gradient rows it will write
        ctx.grads_cleared = any(ctx.needs_input_grad[1:5])
        # construct_dense_sparse_mapping + forward (raycast_rgbd.py:23,26-28) as one native call
        raycast_rgbd_cuda.forward(sparse_mapping.to(device), locs.to(device), vals_sdf, vals_colors, vals_normals,
                                  vals_semantic, view_matrix_inv, image_color, image_depth, image_normal,
                                  image_semantic, mapping3dto2d, mapping3dto2d_num, intrinsic_params, opts,
                                  views_per_chunk=views_per_chunk, flags=flags, build_index=True,
                                  clear_grads=(d_color, d_depth, d_normal, d_semantic) if ctx.grads_cleared else None,
                                  workspace_owner=workspace_owner)
        ctx.workspace_owner = workspace_owner
        ctx.forward_id = None if workspace_owner is None else workspace_owner.forwards
        ctx.flags = flags
        ctx.dims = [sparse_mapping.shape[0], dims3d[2], dims3d[1], dims3d[0], num_locs]  # raycast_rgbd.py:30-31
        ctx.views_per_chunk = views_per_chunk
        ctx.save_for_backward(sparse_mapping, mapping3dto2d, mapping3dto2d_num, d_color, d_depth, d_normal,
                              d_semantic)
        images = sparse_mapping.shape[0] * views_per_chunk
        if images == image_depth.shape[0]:
            return image_color, image_depth, image_normal, image_semantic
        return image_color[:images], image_depth[:images], image_normal[:images], image_semantic[:images]

    @staticmethod
    def _normal_grad(ctx, d_normal, n):
        if ctx.flags & N.SPSG_FLAG_VIEW_NORMALS:
            return d_normal[:n * ctx.views_per_chunk].view(n, ctx.views_per_chunk, 3)
        return d_normal[:n]

    @staticmethod
    def backward(ctx, grad_color, grad_depth, grad_normal, grad_semantic):
        sparse_mapping, mapping3dto2d, mapping3dto2d_num, d_color, d_depth, d_normal, d_semantic = ctx.saved_tensors
        n = ctx.dims[4]
        owner = ctx.workspace_owner
        if owner is not None:
            owner.check_latest(ctx.forward_id)
        raycast_rgbd_cuda.backward(
            grad_color.contiguous(), grad_depth.contiguous(), grad_normal.contiguous(), grad_semantic.contiguous(),
            sparse_mapping, mapping3dto2d, mapping3dto2d_num, ctx.dims, d_color, d_depth, d_normal, d_semantic,
            views_per_chunk=ctx.views_per_chunk, grads_cleared=ctx.grads_cleared, workspace_owner=owner,
            flags=ctx.flags)
        ctx.grads_cleared = False  # the forward cleared the rows once: a second backward (retain_graph) clears its own
        grads = (d_depth[:n], d_color[:n], RayCastRGBDFunction._normal_grad(ctx, d_normal, n), d_semantic[:n])
        if owner is not None:
            owner.grad_views = grads  # leaves get copies, not the buffers (ModuleWorkspace)
        # raycast_rgbd.py:42-43: (locs, vals_sdf, vals_colors, vals_normals, vals_semantic, None...)
        return (None,) + grads + (None,) * (len(ctx.needs_input_grad) - 5)


class RaycastRGBD(nn.Module):
    def __init__(self, batch_size, dims3d, width, height, depth_min, depth_max, thresh_sample_dist, ray_increment,
                 max_num_frames=1, max_num_locs_per_sample=200000, max_pixels_per_voxel=64, device=None, num_classes=14):
        super(RaycastRGBD, self).__init__()
        if not torch.cuda.is_available():
            raise RuntimeError("RaycastRGBD needs a CUDA device: this implementation has no CPU path")
        device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.batch_size = batch_size
        self.max_num_frames = max_num_frames
        self.dims3d = dims3d
        self.width = width
        self.height = height
        self.depth_min = depth_min
        self.depth_max = depth_max
        self.thresh_sample_dist = thresh_sample_dist
        self.ray_increment = ray_increment
        self.max_num_locs_per_sample = max_num_locs_per_sample
        if not 1 <= num_classes <= N.SPSG_MAX_SEMANTIC_CHANNELS:
            raise RuntimeError("num_classes must be in 1..%d, got %d" % (N.SPSG_MAX_SEMANTIC_CHANNELS, num_classes))
        self.num_classes = num_classes
        images = batch_size * max_num_frames
        rows = batch_size * max_num_frames * max_num_locs_per_sample
        # same buffers, shapes and dtypes as raycast_rgbd.py:59-72, allocated directly on the device
        self.image_depth = torch.zeros(images, height, width, device=device)
        self.image_normal = torch.zeros(images, height, width, 3, device=device)
        self.image_color = torch.zeros(images, height, width, 3, device=device)
        self.image_semantic = torch.zeros(images, height, width, num_classes, device=device)
        # max_pixels_per_voxel=None: every pixel of a (voxel, view) enters its gradient (SPSG_FLAG_ALL_PIXELS), no table
        self.mapping3dto2d = torch.zeros(rows, max_pixels_per_voxel, dtype=torch.int, device=device) \
            if max_pixels_per_voxel is not None else torch.empty(0, dtype=torch.int, device=device)
        self.mapping3dto2d_num = torch.zeros(rows, dtype=torch.int, device=device)
        self.sparse_mapping = torch.zeros(batch_size, dims3d[0], dims3d[1], dims3d[2], dtype=torch.int, device=device)
        self.d_color = torch.zeros(batch_size * max_num_locs_per_sample, 3, device=device)
        self.d_normal = torch.zeros(batch_size * max_num_locs_per_sample, 3, device=device)
        self.d_depth = torch.zeros(batch_size * max_num_locs_per_sample, 1, device=device)
        self.d_semantic = torch.zeros(batch_size * max_num_locs_per_sample, num_classes, device=device)
        self.d_normal_views = None  # (N*F,3) gradient rows of per-view normals (raycast_rgbd_cuda.normal_grad_buffer)
        # SPSG_FLAG_* (e.g. _native.SPSG_FLAG_DETERMINISTIC for bit-reproducible tables, losses and gradients; it is also on
        # whenever torch.use_deterministic_algorithms(True) is).  SPSG_FLAG_ALL_PIXELS marks the module without a table:
        # keep it when adding flags (``m.flags |= ...``)
        self.flags = N.SPSG_FLAG_ALL_PIXELS if max_pixels_per_voxel is None else 0
        # scratch of the native calls (block maps, the backward's work list): owned by the module like the buffers above
        self.workspace = raycast_rgbd_cuda.ModuleWorkspace()

    def get_max_num_locs_per_sample(self):
        return self.max_num_locs_per_sample

    def forward(self, locs, vals_sdf, vals_colors, vals_normals, vals_semantics, view_matrix, intrinsic_params):
        if vals_semantics is None:
            vals_semantics = torch.zeros(vals_sdf.shape[0], self.num_classes, device=vals_sdf.device)  # unlabeled class
        elif self.num_classes != 14 and (vals_semantics.dim() != 2 or vals_semantics.shape[1] != self.num_classes):
            # (at 14 the reference's behaviour stays: any payload with at least 14 * N values is read as (N,14))
            raise RuntimeError("vals_semantics must be (N, %d), got %s" % (self.num_classes, tuple(vals_semantics.shape)))
        images = view_matrix.shape[0]
        views = max(1, images // self.batch_size)
        if images != views * self.batch_size or views > self.max_num_frames:
            raise RuntimeError("view_matrix has %d images: expected batch_size (%d) x views with views <= "
                               "max_num_frames (%d)" % (images, self.batch_size, self.max_num_frames))
        per_view = raycast_rgbd_cuda.view_normals(vals_normals, views)
        flags = self.flags | (N.SPSG_FLAG_VIEW_NORMALS if per_view else 0)
        return RayCastRGBDFunction.apply(locs, vals_sdf, vals_colors, vals_normals, vals_semantics, view_matrix,
                                         intrinsic_params, self.dims3d, self.width, self.height, self.depth_min,
                                         self.depth_max, self.thresh_sample_dist, self.ray_increment, self.image_color,
                                         self.image_depth, self.image_normal, self.image_semantic, self.sparse_mapping,
                                         self.mapping3dto2d, self.mapping3dto2d_num, self.d_color, self.d_depth,
                                         raycast_rgbd_cuda.normal_grad_buffer(self, per_view), self.d_semantic, views,
                                         flags, self.workspace)

    def render_labels(self, locs, vals_sdf, voxel_labels, view_matrix, intrinsic_params, histogram=False):
        """The label map of a render, without rendering the semantic image: a new (I,H,W) uint8 tensor holding the hit
        voxel's label (``voxel_labels``, (N,) uint8; a label above ``num_classes`` counts as ``num_classes``), or
        ``num_classes`` where the ray hits nothing.  Same march and hit voxels as ``forward``, so it equals
        ``losses.labels_from_render`` of a forward with the one-hot of ``voxel_labels`` as semantic payload.  With
        ``histogram=True`` also returns the (num_classes + 1,) int64 pixel count per label.  The module's images, tables
        and gradient buffers are not touched; it counts as a forward on the module's workspace, so a backward of an earlier
        forward raises afterwards.  No autograd."""
        images = view_matrix.shape[0]
        views = max(1, images // self.batch_size)
        if images != views * self.batch_size or views > self.max_num_frames:
            raise RuntimeError("view_matrix has %d images: expected batch_size (%d) x views with views <= "
                               "max_num_frames (%d)" % (images, self.batch_size, self.max_num_frames))
        opts = [self.width, self.height, self.depth_min, self.depth_max, self.thresh_sample_dist, self.ray_increment,
                self.dims3d[2], self.dims3d[1], self.dims3d[0]]
        return raycast_rgbd_cuda.render_labels(self.sparse_mapping, locs, vals_sdf, voxel_labels, view_matrix,
                                               intrinsic_params, opts, self.num_classes, views, self.flags, histogram,
                                               self.workspace)


class RaycastOcc(nn.Module):
    def __init__(self, batch_size, dims3d, width, height, depth_min, depth_max, ray_increment, device=None):
        super(RaycastOcc, self).__init__()
        if not torch.cuda.is_available():
            raise RuntimeError("RaycastOcc needs a CUDA device: this implementation has no CPU path")
        device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.dims3d = dims3d
        self.width = width
        self.height = height
        self.depth_min = depth_min
        self.depth_max = depth_max
        self.ray_increment = ray_increment
        self.occ2d = torch.zeros(batch_size, 1, height, width, dtype=torch.uint8, device=device)

    def forward(self, occ3d, view_matrix, intrinsic_params):
        opts = [self.width, self.height, self.depth_min, self.depth_max, self.ray_increment, self.dims3d[2],
                self.dims3d[1], self.dims3d[0]]  # raycast_rgbd.py:100-102
        raycast_rgbd_cuda.raycast_occ(occ3d, self.occ2d, view_matrix, intrinsic_params, opts)
        return self.occ2d
