"""Drop-in for the reference's native extension module ``raycast_rgbd_cuda``.

Same four entry points, positional tensors, in-place outputs and error behaviour as
``torch/utils/raycast_rgbd/raycast_rgbd_cuda.cpp:57-160`` -- but each is a thin adapter
(tensor -> device pointer, current device + stream) over the C ABI of ``include/spsg_raycast.h``.

    forward(sparse_mapping, locs, vals_sdf, vals_color, vals_normals, vals_semantic, viewMatrixInv,
            imageColor, imageDepth, imageNormal, imageSemantic, mapping3dto2d, mapping3dto2d_num,
            intrinsicParams, opts)
    backward(grad_color, grad_depth, grad_normal, grad_semantic, sparse_mapping, mapping3dto2d,
             mapping3dto2d_num, dims, d_color, d_depth, d_normals, d_semantic)
    construct_dense_sparse_mapping(locs, sparse_mapping)
    raycast_occ(occ3d, occ2d, viewMatrixInv, intrinsicParams, opts)
"""
import ctypes
from collections import OrderedDict

import os
import weakref

import torch

from . import _native as N

_MIN_TORCH = (2, 1)
if tuple(int(x) for x in torch.__version__.split("+")[0].split(".")[:2]) < _MIN_TORCH:
    raise ImportError("spsg_b200 needs torch >= %d.%d (found %s)" % (_MIN_TORCH + (torch.__version__,)))

# Workspaces of callers that hold no module (the reference's wrapper talks to this module with bare tensors): strong
# references keyed by the raycaster's `sparse_mapping` buffer, least recently used first, each stamped with the forward
# that filled it.  `RaycastRGBD` (raycast_rgbd.py) and the fused losses pass their own workspace explicitly instead.
_MAX_CACHED_WORKSPACES = 32
_workspaces = OrderedDict()


def _check_input(t, name):
    # CHECK_CUDA / CHECK_CONTIGUOUS (raycast_rgbd_cuda.cpp:53-55): AT_ASSERTM -> RuntimeError
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError("%s must be a CUDA tensor" % name)
    if not t.is_contiguous():
        raise RuntimeError("%s must be contiguous" % name)


def _check_dtype(t, dtype, name):
    if t.dtype != dtype:
        raise RuntimeError("%s must have dtype %s, got %s" % (name, dtype, t.dtype))


def check_voxel_inputs(locs, vals_sdf, vals_color, vals_normals, vals_semantic, view_matrix, intrinsic_params, images,
                       normal_views=1):
    """What every raw-pointer entry point relies on: CUDA + contiguous, int64 `locs` rows of 4, float32 payloads with at
    least N rows of 1 / 3 / 3 / 14 (normals: N * ``normal_views`` rows of 3 with SPSG_FLAG_VIEW_NORMALS), cameras for every
    image.  Raises RuntimeError like the reference's AT_ASSERTM."""
    for t, name in ((locs, "locs"), (vals_sdf, "vals_sdf"), (vals_color, "vals_color"), (vals_normals, "vals_normals"),
                    (vals_semantic, "vals_semantic"), (view_matrix, "viewMatrixInv"), (intrinsic_params, "intrinsicParams")):
        _check_input(t, name)
    if not is_packed_locs(locs):
        _check_dtype(locs, torch.int64, "locs")
    for t, name in ((vals_sdf, "vals_sdf"), (vals_color, "vals_color"), (vals_normals, "vals_normals"),
                    (vals_semantic, "vals_semantic"), (view_matrix, "viewMatrixInv"), (intrinsic_params, "intrinsicParams")):
        _check_dtype(t, torch.float32, name)
    n = locs.shape[0]
    if not is_packed_locs(locs) and locs.numel() != 4 * n:
        raise RuntimeError("locs must be (N, 4) rows of (z, y, x, chunk)")
    if vals_sdf.numel() < n or vals_color.numel() < 3 * n or vals_normals.numel() < 3 * n * normal_views or \
            vals_semantic.numel() < 14 * n:
        raise RuntimeError("voxel value tensors hold fewer than N = %d rows" % n)
    if view_matrix.numel() < images * 16 or intrinsic_params.numel() < images * 4:
        raise RuntimeError("viewMatrixInv / intrinsicParams hold fewer than %d images" % images)
    devs = {t.device for t in (locs, vals_sdf, vals_color, vals_normals, vals_semantic, view_matrix, intrinsic_params)}
    if len(devs) != 1:
        raise RuntimeError("raycast inputs live on different devices: %s" % sorted(str(d) for d in devs))
    return n


def is_packed_locs(locs):
    """``locs`` given as one linear cell index per voxel, (N,) int32 holding uint32 bits -- the output of ``pack_locs_host``
    after its trip over PCIe -- instead of the reference's (N,4) int64 rows."""
    return locs.dim() == 1 and locs.dtype == torch.int32


def pack_locs_host(locs, num_chunks, dims3d, out=None, threads=0):
    """Host side of a host-fed call: the reference's (N,4) int64 (z,y,x,b) rows, in host memory, as one uint32 linear cell
    index each (``spsg_pack_locs_host``): 4 instead of 32 bytes per voxel to carry over PCIe.  ``out``: (N,) int32 CPU tensor to
    write (e.g. a view of the pinned staging buffer); returned.  Pass its device copy as ``locs`` to the forward.
    ``threads`` 0 = the CPUs this process may run on (at most 16)."""
    if locs.device.type != "cpu" or locs.dtype != torch.int64 or not locs.is_contiguous() or locs.dim() != 2 or locs.shape[1] != 4:
        raise RuntimeError("pack_locs_host takes a contiguous (N,4) int64 CPU tensor")
    n = locs.shape[0]
    if out is None:
        out = torch.empty(n, dtype=torch.int32)
    if out.device.type != "cpu" or out.dtype != torch.int32 or not out.is_contiguous() or out.numel() != n:
        raise RuntimeError("out must be a contiguous (N,) int32 CPU tensor")
    if threads <= 0:
        threads = min(16, len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))
    N.check(N.lib.spsg_pack_locs_host(locs.data_ptr(), n, int(num_chunks), int(dims3d[0]), int(dims3d[1]), int(dims3d[2]),
                                      out.data_ptr(), int(threads)))
    return out


def view_normals(vals_normals, views):
    """Normal payload mode of a render with ``views`` images per chunk: False for the shared ``(N,3)`` payload, True for
    per-view normals ``(N,views,3)`` (SPSG_FLAG_VIEW_NORMALS; the gradient is ``(N,views,3)`` too)."""
    if vals_normals.dim() != 3:
        return False
    if vals_normals.shape[1] != views or vals_normals.shape[2] != 3:
        raise RuntimeError("per-view vals_normals must be (N, %d, 3) for %d views per chunk, got %s"
                           % (views, views, tuple(vals_normals.shape)))
    return True


def normal_grad_buffer(m, per_view):
    """The ``d_normal`` rows a backward of raycaster ``m`` writes: ``m.d_normal`` (N,3), or with per-view normals a
    separate buffer of ``m.d_normal.shape[0] * m.max_num_frames`` rows, allocated on first use."""
    if not per_view:
        return m.d_normal
    buf = getattr(m, "d_normal_views", None)
    if buf is None:
        buf = m.d_normal_views = torch.zeros(m.d_normal.shape[0] * m.max_num_frames, 3, device=m.d_normal.device)
    return buf


def with_torch_mode(flags):
    """``flags`` plus SPSG_FLAG_DETERMINISTIC while ``torch.use_deterministic_algorithms(True)`` is in effect: every raycast
    and 2D-loss call then gives results that depend on its inputs alone (canonical voxel -> pixel tables, loss sums in pixel
    order, no float atomics).  Read at each call, forward and backward alike."""
    return flags | N.SPSG_FLAG_DETERMINISTIC if torch.are_deterministic_algorithms_enabled() else flags


def _stamp(p):
    return (int(p.num_locs), int(p.views_per_chunk), int(p.num_chunks), int(p.width), int(p.height),
            int(p.max_pixels_per_voxel), bool(p.flags & N.SPSG_FLAG_VIEW_NORMALS),
            "deterministic" if p.flags & N.SPSG_FLAG_DETERMINISTIC else "default")


def workspace(device, nbytes, owner=None, stamp=None, expect=None):
    """Scratch tensor for callers without a module, keyed by the raycaster's ``sparse_mapping`` buffer and grown on demand;
    the C ABI never allocates.  The forward leaves the backward's work list in it and records ``stamp`` (what it was run
    with); the backward passes ``expect`` and gets an error -- not garbage -- if no forward with those parameters filled
    the workspace of this raycaster."""
    key = (device.type, device.index, None if owner is None else owner.data_ptr())
    entry = _workspaces.get(key)
    if expect is not None:
        if entry is None or entry["stamp"] != expect or entry["ws"].numel() < nbytes:
            raise RuntimeError("raycast backward without a matching forward on these buffers (forward ran with %s, backward "
                               "asks for %s)" % (None if entry is None else entry["stamp"], expect))
        _workspaces.move_to_end(key)
        return entry["ws"]
    if entry is None or entry["ws"].numel() < nbytes:
        entry = {"ws": torch.empty(max(int(nbytes), 1 << 16), dtype=torch.uint8, device=device), "stamp": None}
        _workspaces[key] = entry
        while len(_workspaces) > _MAX_CACHED_WORKSPACES:
            _workspaces.popitem(last=False)
    _workspaces.move_to_end(key)
    if stamp is not None:
        entry["stamp"] = stamp
    return entry["ws"]


class ModuleWorkspace:
    """The workspace of one raycaster module: an explicit buffer it owns, stamped by every forward.

    ``forwards`` counts the forwards that filled it: an autograd backward records the count its forward left and refuses
    to gather once a later forward has overwritten the module's tables and images (``check_latest``).  ``grad_views``
    holds the ``d_*`` row views the last autograd backward returned: with that extra reference, autograd copies them into
    the ``.grad`` of leaf tensors instead of storing the module's buffers there (which the next forward clears)."""

    def __init__(self):
        self.ws, self.stamp, self._prebuilt = None, None, None
        self.forwards = 0
        self.grad_views = None

    def get(self, device, nbytes):
        if self.ws is None or self.ws.numel() < nbytes or self.ws.device != device:
            self.ws = torch.empty(max(int(nbytes), 1 << 16), dtype=torch.uint8, device=device)
            self.stamp, self._prebuilt = None, None
        return self.ws

    # The voxel index and the dense SDF brick can be written together with ``locs`` (sparsify.sparsify_predictions(...,
    # raycaster=m)); the forward that renders exactly that ``locs`` tensor then skips its fill and index passes.  Any other
    # forward on the module overwrites them, which drops the mark.
    def mark_prebuilt(self, locs):
        self._prebuilt = (weakref.ref(locs), locs._version, locs.shape[0])

    def take_prebuilt(self, locs, nbytes):
        """SPSG_FLAG_INDEX_PREBUILT if index + brick in this workspace belong to ``locs`` (same tensor object, unmodified), else
        0; either way the mark is re-derived by the caller after the forward."""
        mark, self._prebuilt = self._prebuilt, None
        if mark is None or self.ws is None or self.ws.numel() < nbytes:
            return 0
        ref, version, n = mark
        return N.SPSG_FLAG_INDEX_PREBUILT if ref() is locs and locs._version == version and locs.shape[0] == n else 0

    def filled(self, p):
        self.stamp = _stamp(p)
        self.forwards += 1

    def check_latest(self, forward):
        """``forward`` = ``self.forwards`` right after the forward whose backward is about to run."""
        if forward != self.forwards:
            raise RuntimeError("raycast backward after a later forward on the same module: that forward overwrote the "
                               "registration tables and renderings this backward gathers from (%d forwards since)"
                               % (self.forwards - forward))

    def check(self, p, nbytes):
        if self.ws is None or self.stamp != _stamp(p) or self.ws.numel() < nbytes:
            raise RuntimeError("raycast backward without a matching forward on this module (forward ran with %s, backward "
                               "asks for %s)" % (self.stamp, _stamp(p)))
        return self.ws


def _stream(device):
    return torch.cuda.current_stream(device).cuda_stream


class _NoGuard:
    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False


_NO_GUARD = _NoGuard()


def device_guard(device):
    """``torch.cuda.device(device)`` only when ``device`` is not already current (the context manager costs ~10 us of
    host time per call, which matters for a 50 us step)."""
    idx = device.index
    if idx is None or idx == torch.cuda.current_device():
        return _NO_GUARD
    return torch.cuda.device(device)


def _opt_int(v):
    return int(float(v) + 0.5)  # raycast_rgbd_cuda_kernel.cu:445-456


def construct_dense_sparse_mapping(locs, sparse_mapping):
    _check_input(locs, "locs")
    _check_input(sparse_mapping, "sparse_mapping")
    _check_dtype(locs, torch.int64, "locs")
    _check_dtype(sparse_mapping, torch.int32, "sparse_mapping")
    with device_guard(sparse_mapping.device):
        N.check(N.lib.spsg_build_index(N.ptr(locs), locs.shape[0], N.ptr(sparse_mapping), sparse_mapping.shape[0],
                                       sparse_mapping.shape[1], sparse_mapping.shape[2], sparse_mapping.shape[3],
                                       _stream(sparse_mapping.device)))


def _forward_params(sparse_mapping, locs, mapping3dto2d, opts, views_per_chunk=1, flags=0):
    o = opts.tolist() if isinstance(opts, torch.Tensor) else list(opts)
    return N.make_params(width=_opt_int(o[0]), height=_opt_int(o[1]), depth_min=o[2], depth_max=o[3],
                         thresh_sample_dist=o[4], ray_increment=o[5], dimx=_opt_int(o[6]), dimy=_opt_int(o[7]),
                         dimz=_opt_int(o[8]), num_chunks=sparse_mapping.shape[0], views_per_chunk=views_per_chunk,
                         max_pixels_per_voxel=mapping3dto2d.shape[1], num_locs=locs.shape[0], flags=flags)


def forward(sparse_mapping, locs, vals_sdf, vals_color, vals_normals, vals_semantic, viewMatrixInv, imageColor,
            imageDepth, imageNormal, imageSemantic, mapping3dto2d, mapping3dto2d_num, intrinsicParams, opts,
            views_per_chunk=1, flags=0, build_index=False, clear_grads=None, workspace_owner=None):
    """Reference signature (``raycast_color_forward``, raycast_rgbd_cuda.cpp:57-91) plus keyword extensions with
    reference-preserving defaults.  ``clear_grads`` = (d_color, d_depth, d_normals, d_semantic) lets the forward's fill
    pass clear the rows the matching ``backward(..., grads_cleared=True)`` will write (needs ``build_index=True``).
    ``flags`` with SPSG_FLAG_VIEW_NORMALS: ``vals_normals`` (and ``d_normals`` of ``clear_grads``) hold N*F rows.
    ``workspace_owner`` = the calling module's ``ModuleWorkspace`` (else the scratch is looked up by ``sparse_mapping``).
    Deterministic mode (SPSG_FLAG_DETERMINISTIC) is on when ``flags`` has it or torch's deterministic algorithms are enabled;
    the matching ``backward`` must run in the same mode."""
    flags = with_torch_mode(flags)
    for t, name in ((sparse_mapping, "sparse_mapping"), (imageColor, "imageColor"), (imageDepth, "imageDepth"),
                    (imageNormal, "imageNormal"), (imageSemantic, "imageSemantic"), (mapping3dto2d, "mapping3dto2d"),
                    (mapping3dto2d_num, "mapping3dto2d_num")):
        _check_input(t, name)
    _check_dtype(sparse_mapping, torch.int32, "sparse_mapping")
    _check_dtype(mapping3dto2d, torch.int32, "mapping3dto2d")
    _check_dtype(mapping3dto2d_num, torch.int32, "mapping3dto2d_num")
    for t, name in ((imageColor, "imageColor"), (imageDepth, "imageDepth"), (imageNormal, "imageNormal"),
                    (imageSemantic, "imageSemantic")):
        _check_dtype(t, torch.float32, name)
    p = _forward_params(sparse_mapping, locs, mapping3dto2d, opts, views_per_chunk, flags)
    if is_packed_locs(locs):
        if not build_index:
            raise RuntimeError("packed locs need build_index=True")
        p.flags |= N.SPSG_FLAG_PACKED_LOCS
    images = p.num_chunks * p.views_per_chunk
    nv = p.views_per_chunk if flags & N.SPSG_FLAG_VIEW_NORMALS else 1
    n = check_voxel_inputs(locs, vals_sdf, vals_color, vals_normals, vals_semantic, viewMatrixInv, intrinsicParams, images,
                           nv)
    if mapping3dto2d_num.numel() < p.views_per_chunk * n or mapping3dto2d.shape[0] < p.views_per_chunk * n:
        raise RuntimeError("mapping3dto2d has %d rows, needs views_per_chunk*N = %d" %
                           (mapping3dto2d.shape[0], p.views_per_chunk * n))
    px = images * p.width * p.height
    if imageDepth.numel() < px or imageColor.numel() < 3 * px or imageNormal.numel() < 3 * px or \
            imageSemantic.numel() < 14 * px:
        raise RuntimeError("image buffers are smaller than %d x %d x %d" % (images, p.height, p.width))
    dev = vals_sdf.device
    with device_guard(dev):
        nbytes = N.workspace_bytes(p)
        if workspace_owner is not None:
            prebuilt = workspace_owner.take_prebuilt(locs, nbytes) if build_index else 0
            ws = workspace_owner.get(dev, nbytes)
            p.flags |= prebuilt
        else:
            ws = workspace(dev, nbytes, sparse_mapping, stamp=_stamp(p))
        args = (ctypes.byref(p), N.ptr(sparse_mapping), N.ptr(locs), N.ptr(vals_sdf), N.ptr(vals_color),
                N.ptr(vals_normals), N.ptr(vals_semantic), N.ptr(viewMatrixInv), N.ptr(intrinsicParams),
                N.ptr(imageColor), N.ptr(imageDepth), N.ptr(imageNormal), N.ptr(imageSemantic),
                N.ptr(mapping3dto2d), N.ptr(mapping3dto2d_num))
        if build_index:
            gb = None
            if clear_grads is not None:
                for t, rows in zip(clear_grads, (3, 1, 3 * nv, 14)):
                    _check_input(t, "clear_grads")
                    _check_dtype(t, torch.float32, "clear_grads")
                    if t.numel() < n * rows:
                        raise RuntimeError("d_* buffers hold fewer than N = %d rows" % n)
                gb = ctypes.byref(N.grad_buffers(*clear_grads))
            N.check(N.lib.spsg_raycast_forward_indexed(*args, gb, N.ptr(ws), ws.numel(), _stream(dev)))
        else:
            if clear_grads is not None:
                raise RuntimeError("clear_grads needs build_index=True")
            N.check(N.lib.spsg_raycast_forward(*args, N.ptr(ws), ws.numel(), _stream(dev)))
        if workspace_owner is not None:
            workspace_owner.filled(p)
            if p.flags & N.SPSG_FLAG_INDEX_PREBUILT:
                workspace_owner.mark_prebuilt(locs)  # index and brick are untouched: still valid for these rows
    return ws


def backward(grad_color, grad_depth, grad_normal, grad_semantic, sparse_mapping, mapping3dto2d, mapping3dto2d_num,
             dims, d_color, d_depth, d_normals, d_semantic, views_per_chunk=1, grads_cleared=False, workspace_owner=None,
             flags=0):
    """Reference signature (``raycast_color_backward``, raycast_rgbd_cuda.cpp:102-140).
    ``dims`` = int32 CPU tensor (or sequence) [batch, Dx, Dy, Dz, N] (raycast_rgbd.py:30-31).  ``flags``: the forward's
    SPSG_FLAG_DETERMINISTIC_GRADS, SPSG_FLAG_VIEW_NORMALS (``d_normals`` then holds N*F rows) and SPSG_FLAG_DETERMINISTIC
    are used; the last is also on under torch's deterministic algorithms, and a backward in another mode than its forward
    raises RuntimeError."""
    flags = with_torch_mode(flags)
    for t, name in ((grad_color, "grad_color"), (grad_depth, "grad_depth"), (grad_normal, "grad_normal"),
                    (grad_semantic, "grad_semantic"), (sparse_mapping, "sparse_mapping"),
                    (mapping3dto2d, "mapping3dto2d"), (mapping3dto2d_num, "mapping3dto2d_num"),
                    (d_color, "d_color"), (d_depth, "d_depth"), (d_normals, "d_normals"), (d_semantic, "d_semantic")):
        _check_input(t, name)
    for t, name in ((grad_color, "grad_color"), (grad_depth, "grad_depth"), (grad_normal, "grad_normal"),
                    (grad_semantic, "grad_semantic"), (d_color, "d_color"), (d_depth, "d_depth"), (d_normals, "d_normals"),
                    (d_semantic, "d_semantic")):
        _check_dtype(t, torch.float32, name)
    d = dims.tolist() if isinstance(dims, torch.Tensor) else list(dims)
    n = int(d[4])
    nv = views_per_chunk if flags & N.SPSG_FLAG_VIEW_NORMALS else 1
    if d_color.shape[0] < n or d_depth.shape[0] < n or d_normals.shape[0] < n * nv or d_semantic.shape[0] < n:
        raise RuntimeError("d_* buffers hold fewer than N = %d rows" % n)
    p = N.make_params(width=grad_color.shape[2], height=grad_color.shape[1], depth_min=0, depth_max=0,
                      thresh_sample_dist=0, ray_increment=0, dimx=int(d[1]), dimy=int(d[2]), dimz=int(d[3]),
                      num_chunks=sparse_mapping.shape[0], views_per_chunk=views_per_chunk,
                      max_pixels_per_voxel=mapping3dto2d.shape[1], num_locs=n,
                      flags=(N.SPSG_FLAG_GRADS_CLEARED if grads_cleared else 0) |
                      (flags & (N.SPSG_FLAG_DETERMINISTIC_GRADS | N.SPSG_FLAG_VIEW_NORMALS | N.SPSG_FLAG_DETERMINISTIC)))
    dev = grad_color.device
    px = sparse_mapping.shape[0] * views_per_chunk * p.width * p.height
    if grad_depth.numel() < px or grad_color.numel() < 3 * px or grad_normal.numel() < 3 * px or grad_semantic.numel() < 14 * px:
        raise RuntimeError("gradient images are smaller than %d x %d x %d" % (px // (p.width * p.height), p.height, p.width))
    with device_guard(dev):
        nbytes = N.workspace_bytes(p)
        # the work list of the forward that rendered these images: refuse to run on anything else
        ws = workspace_owner.check(p, nbytes) if workspace_owner is not None else \
            workspace(dev, nbytes, sparse_mapping, expect=_stamp(p))
        N.check(N.lib.spsg_raycast_backward(ctypes.byref(p), N.ptr(grad_color), N.ptr(grad_depth), N.ptr(grad_normal),
                                            N.ptr(grad_semantic), N.ptr(sparse_mapping), N.ptr(mapping3dto2d),
                                            N.ptr(mapping3dto2d_num), N.ptr(d_color), N.ptr(d_depth),
                                            N.ptr(d_normals), N.ptr(d_semantic), N.ptr(ws), ws.numel(), _stream(dev)))


def raycast_occ(occ3d, occ2d, viewMatrixInv, intrinsicParams, opts, flags=0):
    """Reference signature (``raycast_occ_forward``, raycast_rgbd_cuda.cpp:142-153);
    opts = [W, H, depth_min, depth_max, ray_increment, ...] (raycast_rgbd_cuda_kernel.cu:596-602)."""
    for t, name in ((occ3d, "occ3d"), (occ2d, "occ2d"), (viewMatrixInv, "viewMatrixInv"),
                    (intrinsicParams, "intrinsicParams")):
        _check_input(t, name)
    _check_dtype(occ3d, torch.uint8, "occ3d")
    _check_dtype(occ2d, torch.uint8, "occ2d")
    o = opts.tolist() if isinstance(opts, torch.Tensor) else list(opts)
    p = N.make_params(width=_opt_int(o[0]), height=_opt_int(o[1]), depth_min=o[2], depth_max=o[3],
                      thresh_sample_dist=0, ray_increment=o[4], dimx=occ3d.shape[4], dimy=occ3d.shape[3],
                      dimz=occ3d.shape[2], num_chunks=occ3d.shape[0], flags=flags)
    dev = occ3d.device
    with device_guard(dev):
        N.check(N.lib.spsg_raycast_occ(ctypes.byref(p), N.ptr(occ3d), N.ptr(occ2d), N.ptr(viewMatrixInv),
                                       N.ptr(intrinsicParams), _stream(dev)))
