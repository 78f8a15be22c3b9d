"""ctypes binding of the C ABI declared in ``include/spsg_raycast.h``.

There is deliberately NO fallback: if ``lib/libspsg_raycast.so`` is missing or fails to load, importing this
module raises, and so does everything built on it.  Build it with ``python -c "import __graft_entry__ as g;
g.build()"`` (or ``make -C <package>/csrc``).
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SPSG_RAYCAST_LIB", os.path.join(_HERE, "lib", "libspsg_raycast.so"))

SPSG_FLAG_NO_CLIP = 1 << 0
SPSG_FLAG_NO_BRICK_SKIP = 1 << 1
SPSG_FLAG_RECORD_HITS = 1 << 2
SPSG_FLAG_GRADS_CLEARED = 1 << 3
SPSG_FLAG_DETERMINISTIC_GRADS = 1 << 4
SPSG_FLAG_SMEM_MAPS = 1 << 5
SPSG_FLAG_GLOBAL_MAPS = 1 << 6
SPSG_FLAG_INDEX_PREBUILT = 1 << 7
SPSG_FLAG_PACKED_LOCS = 1 << 8
SPSG_FLAG_VIEW_NORMALS = 1 << 9
SPSG_FLAG_DETERMINISTIC = 1 << 10
SPSG_FLAG_ALL_PIXELS = 1 << 11
SPSG_FLAG_GENERIC_SEMANTIC = 1 << 12
SPSG_MAX_SEMANTIC_CHANNELS = 64
SPSG_LOSS_OUT_FLOATS = 8
SPSG_DTYPE_F32 = 0
SPSG_DTYPE_BF16 = 1
SPSG_DEPTH_MAX_FILL_ROUNDS = 64

# every symbol include/spsg_raycast.h declares (tests check the library exports them all)
EXPORTS = (
    "spsg_version", "spsg_last_error", "spsg_workspace_bytes", "spsg_build_index", "spsg_raycast_forward",
    "spsg_raycast_forward_indexed", "spsg_raycast_backward", "spsg_raycast_occ", "spsg_raycast_forward_loss",
    "spsg_raycast_backward_loss", "spsg_raycast_backward_loss_upstream", "spsg_timing_enable", "spsg_timing_read",
    "spsg_normals_forward", "spsg_normals_backward", "spsg_normals_forward_views", "spsg_normals_backward_views",
    "spsg_losses2d_forward", "spsg_losses2d_backward", "spsg_losses2d_deterministic_scratch_bytes",
    "spsg_losses2d_forward_deterministic",
    "spsg_depth_bilateral_filter", "spsg_depth_median_fill", "spsg_depth_to_cameraspace", "spsg_depth_to_normals",
    "spsg_depth_compute_normals",
    "spsg_sparsify_scratch_bytes", "spsg_sparsify_count", "spsg_sparsify_locs", "spsg_sparsify_locs_indexed",
    "spsg_dense_gather", "spsg_dense_scatter",
    "spsg_sparsify_count_bf16", "spsg_sparsify_locs_bf16", "spsg_sparsify_locs_indexed_bf16",
    "spsg_dense_gather_strided", "spsg_dense_scatter_strided",
    "spsg_labels_from_render", "spsg_pack_locs_host",
    "spsg_losses2d_forward_classes", "spsg_losses2d_forward_deterministic_classes", "spsg_losses2d_backward_classes",
    "spsg_labels_from_render_classes", "spsg_raycast_labels", "spsg_raycast_eval", "spsg_raycast_eval_scratch_bytes",
)


class Params(ctypes.Structure):
    """``spsg_raycast_params``"""
    _fields_ = [
        ("width", ctypes.c_int32), ("height", ctypes.c_int32),
        ("depth_min", ctypes.c_float), ("depth_max", ctypes.c_float),
        ("thresh_sample_dist", ctypes.c_float), ("ray_increment", ctypes.c_float),
        ("dimx", ctypes.c_int32), ("dimy", ctypes.c_int32), ("dimz", ctypes.c_int32),
        ("num_chunks", ctypes.c_int32), ("views_per_chunk", ctypes.c_int32),
        ("max_pixels_per_voxel", ctypes.c_int32),
        ("num_locs", ctypes.c_int64),
        ("flags", ctypes.c_uint32), ("semantic_channels", ctypes.c_uint32),
    ]


class LossTargets(ctypes.Structure):
    """``spsg_loss_targets``"""
    _fields_ = [
        ("target_depth", ctypes.c_void_p), ("target_color", ctypes.c_void_p), ("weight_color", ctypes.c_void_p),
        ("target_label", ctypes.c_void_p), ("class_weight", ctypes.c_void_p),
        ("voxelsize", ctypes.c_float), ("weight_depth", ctypes.c_float), ("weight_color_loss", ctypes.c_float),
        ("weight_semantic", ctypes.c_float),
    ]


class DensePayload(ctypes.Structure):
    """``spsg_dense_payload``"""
    _fields_ = [("dense", ctypes.c_void_p), ("sparse", ctypes.c_void_p), ("channels", ctypes.c_int32),
                ("reserved", ctypes.c_int32)]


class DenseHead(ctypes.Structure):
    """``spsg_dense_head``"""
    _fields_ = [("dense", ctypes.c_void_p), ("sparse", ctypes.c_void_p), ("strides", ctypes.c_int64 * 5),
                ("extent", ctypes.c_int64), ("channels", ctypes.c_int32), ("dtype", ctypes.c_int32)]


class GradBuffers(ctypes.Structure):
    """``spsg_grad_buffers``"""
    _fields_ = [("d_color", ctypes.c_void_p), ("d_depth", ctypes.c_void_p), ("d_normal", ctypes.c_void_p),
                ("d_semantic", ctypes.c_void_p)]


class UpstreamGrads(ctypes.Structure):
    """``spsg_upstream_grads``"""
    _fields_ = [("grad_color", ctypes.c_void_p), ("grad_depth", ctypes.c_void_p), ("grad_normal", ctypes.c_void_p),
                ("grad_semantic", ctypes.c_void_p)]


def _load():
    if not os.path.isfile(LIB_PATH):
        raise ImportError(
            "spsg_b200: CUDA library %s not found -- build it first (python -c 'import __graft_entry__ as g; "
            "g.build()').  There is no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    vp, i32, i64, sz = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_size_t
    pp = ctypes.POINTER(Params)
    lt = ctypes.POINTER(LossTargets)
    lib.spsg_version.restype = ctypes.c_char_p
    lib.spsg_version.argtypes = []
    lib.spsg_last_error.restype = ctypes.c_char_p
    lib.spsg_last_error.argtypes = []
    lib.spsg_workspace_bytes.restype = sz
    lib.spsg_workspace_bytes.argtypes = [pp]
    lib.spsg_build_index.restype = ctypes.c_int
    lib.spsg_build_index.argtypes = [vp, i64, vp, i32, i32, i32, i32, vp]
    gb = ctypes.POINTER(GradBuffers)
    lib.spsg_raycast_forward.restype = ctypes.c_int
    lib.spsg_raycast_forward.argtypes = [pp] + [vp] * 14 + [vp, sz, vp]
    lib.spsg_raycast_forward_indexed.restype = ctypes.c_int
    lib.spsg_raycast_forward_indexed.argtypes = [pp] + [vp] * 14 + [gb, vp, sz, vp]
    lib.spsg_raycast_labels.restype = ctypes.c_int
    lib.spsg_raycast_labels.argtypes = [pp] + [vp] * 8 + [vp, sz, vp]
    lib.spsg_raycast_eval.restype = ctypes.c_int
    lib.spsg_raycast_eval.argtypes = [pp] + [vp] * 8 + [lt, vp, vp, vp, vp, sz, vp, sz, vp]
    lib.spsg_raycast_eval_scratch_bytes.restype = sz
    lib.spsg_raycast_eval_scratch_bytes.argtypes = [pp]
    lib.spsg_raycast_backward.restype = ctypes.c_int
    lib.spsg_raycast_backward.argtypes = [pp] + [vp] * 11 + [vp, sz, vp]
    lib.spsg_raycast_occ.restype = ctypes.c_int
    lib.spsg_raycast_occ.argtypes = [pp, vp, vp, vp, vp, vp]
    lib.spsg_raycast_forward_loss.restype = ctypes.c_int
    lib.spsg_raycast_forward_loss.argtypes = [pp] + [vp] * 14 + [lt, vp, gb, vp, sz, vp]
    lib.spsg_raycast_backward_loss.restype = ctypes.c_int
    lib.spsg_raycast_backward_loss.argtypes = [pp, vp, vp, vp, lt, vp, vp] + [vp] * 7 + [vp, sz, vp]
    lib.spsg_raycast_backward_loss_upstream.restype = ctypes.c_int
    lib.spsg_raycast_backward_loss_upstream.argtypes = [pp, vp, vp, vp, lt, vp, vp, ctypes.POINTER(UpstreamGrads)] + \
        [vp] * 7 + [vp, sz, vp]
    lib.spsg_normals_forward.restype = ctypes.c_int
    lib.spsg_normals_forward.argtypes = [vp, i64, vp, vp, vp, i32, i32, i32, i32, vp, vp]
    lib.spsg_normals_backward.restype = ctypes.c_int
    lib.spsg_normals_backward.argtypes = [vp, i64, vp, vp, vp, i32, i32, i32, i32, vp, vp, vp, vp]
    lib.spsg_normals_forward_views.restype = ctypes.c_int
    lib.spsg_normals_forward_views.argtypes = [vp, i64, vp, vp, i32, vp, i32, i32, i32, i32, vp, vp]
    lib.spsg_normals_backward_views.restype = ctypes.c_int
    lib.spsg_normals_backward_views.argtypes = [vp, i64, vp, vp, i32, vp, i32, i32, i32, i32, vp, vp, vp, vp]
    lib.spsg_losses2d_forward.restype = ctypes.c_int
    lib.spsg_losses2d_forward.argtypes = [lt, vp, vp, vp, i64, vp, vp, sz, vp]
    lib.spsg_losses2d_deterministic_scratch_bytes.restype = sz
    lib.spsg_losses2d_deterministic_scratch_bytes.argtypes = [i64]
    lib.spsg_losses2d_forward_deterministic.restype = ctypes.c_int
    lib.spsg_losses2d_forward_deterministic.argtypes = [lt, vp, vp, vp, i64, vp, vp, sz, vp]
    lib.spsg_losses2d_backward.restype = ctypes.c_int
    lib.spsg_losses2d_backward.argtypes = [lt, vp, vp, vp, i64, vp, vp, vp, vp, vp, vp]
    lib.spsg_losses2d_forward_classes.restype = ctypes.c_int
    lib.spsg_losses2d_forward_classes.argtypes = [lt, vp, vp, vp, i32, i64, vp, vp, sz, vp]
    lib.spsg_losses2d_forward_deterministic_classes.restype = ctypes.c_int
    lib.spsg_losses2d_forward_deterministic_classes.argtypes = [lt, vp, vp, vp, i32, i64, vp, vp, sz, vp]
    lib.spsg_losses2d_backward_classes.restype = ctypes.c_int
    lib.spsg_losses2d_backward_classes.argtypes = [lt, vp, vp, vp, i32, i64, vp, vp, vp, vp, vp, vp]
    f32 = ctypes.c_float
    lib.spsg_depth_bilateral_filter.restype = ctypes.c_int
    lib.spsg_depth_bilateral_filter.argtypes = [vp, vp, i32, i32, i32, f32, f32, vp]
    lib.spsg_depth_median_fill.restype = ctypes.c_int
    lib.spsg_depth_median_fill.argtypes = [vp, vp, i32, i32, i32, vp]
    lib.spsg_depth_to_cameraspace.restype = ctypes.c_int
    lib.spsg_depth_to_cameraspace.argtypes = [vp, vp, vp, i32, i32, i32, vp]
    lib.spsg_depth_compute_normals.restype = ctypes.c_int
    lib.spsg_depth_compute_normals.argtypes = [vp, vp, i32, i32, i32, vp]
    lib.spsg_depth_to_normals.restype = ctypes.c_int
    lib.spsg_depth_to_normals.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, i32, f32, f32, i32, vp]
    dp = ctypes.POINTER(DensePayload)
    lib.spsg_sparsify_scratch_bytes.restype = sz
    lib.spsg_sparsify_scratch_bytes.argtypes = [i64]
    lib.spsg_sparsify_count.restype = ctypes.c_int
    lib.spsg_sparsify_count.argtypes = [vp, vp, i64, f32, vp, sz, vp, vp]
    lib.spsg_sparsify_locs.restype = ctypes.c_int
    lib.spsg_sparsify_locs.argtypes = [vp, vp, i32, i32, i32, i32, f32, vp, vp, i64, vp]
    lib.spsg_pack_locs_host.restype = ctypes.c_int
    lib.spsg_pack_locs_host.argtypes = [vp, i64, i32, i32, i32, i32, vp, i32]
    lib.spsg_sparsify_locs_indexed.restype = ctypes.c_int
    lib.spsg_sparsify_locs_indexed.argtypes = [vp, vp, i32, i32, i32, i32, f32, vp, vp, i64, vp, vp, vp]
    lib.spsg_dense_gather.restype = ctypes.c_int
    lib.spsg_dense_gather.argtypes = [dp, i32, vp, i64, i32, i32, i32, i32, vp]
    lib.spsg_dense_scatter.restype = ctypes.c_int
    lib.spsg_dense_scatter.argtypes = [dp, i32, vp, i64, i32, i32, i32, i32, vp]
    lib.spsg_sparsify_count_bf16.restype = ctypes.c_int
    lib.spsg_sparsify_count_bf16.argtypes = [vp, vp, i64, f32, vp, sz, vp, vp]
    lib.spsg_sparsify_locs_bf16.restype = ctypes.c_int
    lib.spsg_sparsify_locs_bf16.argtypes = [vp, vp, i32, i32, i32, i32, f32, vp, vp, i64, vp]
    lib.spsg_sparsify_locs_indexed_bf16.restype = ctypes.c_int
    lib.spsg_sparsify_locs_indexed_bf16.argtypes = [vp, vp, i32, i32, i32, i32, f32, vp, vp, i64, vp, vp, vp]
    dh = ctypes.POINTER(DenseHead)
    lib.spsg_dense_gather_strided.restype = ctypes.c_int
    lib.spsg_dense_gather_strided.argtypes = [dh, i32, vp, i64, i32, i32, i32, i32, vp]
    lib.spsg_dense_scatter_strided.restype = ctypes.c_int
    lib.spsg_dense_scatter_strided.argtypes = [dh, i32, vp, i64, i32, i32, i32, i32, vp]
    lib.spsg_labels_from_render.restype = ctypes.c_int
    lib.spsg_labels_from_render.argtypes = [vp, i64, vp, vp, vp]
    lib.spsg_labels_from_render_classes.restype = ctypes.c_int
    lib.spsg_labels_from_render_classes.argtypes = [vp, i32, i64, vp, vp, vp]
    lib.spsg_timing_enable.restype = None
    lib.spsg_timing_enable.argtypes = [ctypes.c_int]
    lib.spsg_timing_read.restype = ctypes.c_int
    lib.spsg_timing_read.argtypes = [ctypes.c_int, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int)]
    return lib


lib = _load()


class SpsgError(RuntimeError):
    pass


def check(rc):
    if rc != 0:
        raise SpsgError("spsg_raycast error %d: %s" % (rc, lib.spsg_last_error().decode("utf-8", "replace")))


def version():
    return lib.spsg_version().decode()


def make_params(width, height, depth_min, depth_max, thresh_sample_dist, ray_increment, dimx, dimy, dimz, num_chunks,
                views_per_chunk=1, max_pixels_per_voxel=64, num_locs=0, flags=0, semantic_channels=0):
    """``semantic_channels``: C, the semantic classes per voxel / pixel (0 = 14)."""
    return Params(int(width), int(height), float(depth_min), float(depth_max), float(thresh_sample_dist),
                  float(ray_increment), int(dimx), int(dimy), int(dimz), int(num_chunks), int(views_per_chunk),
                  int(max_pixels_per_voxel), int(num_locs), int(flags), int(semantic_channels))


def workspace_bytes(params):
    n = lib.spsg_workspace_bytes(ctypes.byref(params))
    if n == 0:
        raise SpsgError("spsg_workspace_bytes: %s" % lib.spsg_last_error().decode("utf-8", "replace"))
    return n


def grad_buffers(d_color, d_depth, d_normal, d_semantic):
    return GradBuffers(d_color.data_ptr(), d_depth.data_ptr(), d_normal.data_ptr(), d_semantic.data_ptr())


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def timing_enable(on):
    lib.spsg_timing_enable(1 if on else 0)


def timing_read(which):
    """(total_ms, launches) of the raycast forward kernel (which=0) / backward gather kernel (which=1) since the last
    read."""
    ms, cnt = ctypes.c_double(0.0), ctypes.c_int(0)
    check(lib.spsg_timing_read(int(which), ctypes.byref(ms), ctypes.byref(cnt)))
    return ms.value, cnt.value
