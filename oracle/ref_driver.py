"""Drive the compiled *reference* extension (oracle/_ref/spsg_ref_raycast_cuda.so) through its own native entry
points, allocating buffers the way the reference's Python wrapper does (raycast_rgbd.py:59-72) and calling
construct_dense_sparse_mapping -> forward -> backward in its order (raycast_rgbd.py:23-28, 39-41).
Where the extensions are not built, a test may ask for the stand-in checked against the reference's recorded outputs
(oracle/ref_pins.py) by passing ``pinned=True``; without it a missing extension is an error.
Test infrastructure only."""
import importlib
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = os.path.join(ROOT, "oracle", "_ref")
RAYCAST_SO = os.path.join(REF_DIR, "spsg_ref_raycast_cuda.so")
DEPTH_SO = os.path.join(REF_DIR, "spsg_ref_depth_utils_cuda.so")
_mods = {}


def available(pinned=False):
    """The compiled reference raycaster is present -- or, with ``pinned``, its recorded outputs (tests only)."""
    from oracle import ref_pins
    return os.path.isfile(RAYCAST_SO) or (pinned and ref_pins.recorded())


def depth_available(pinned=False):
    from oracle import ref_pins
    return os.path.isfile(DEPTH_SO) or (pinned and ref_pins.recorded())


def _module(kind, so, pinned):
    from oracle import ref_pins
    built = os.path.isfile(so)
    if not built and not pinned:
        raise ImportError("%s is not built (run __graft_entry__.build() where the reference sources exist)" % so)
    key = (kind, built)
    if key not in _mods:
        if built:
            if REF_DIR not in sys.path:
                sys.path.insert(0, REF_DIR)
            impl = importlib.import_module(os.path.basename(so)[:-3])
            _mods[key] = ref_pins.PinnedModule(impl, kind, record=True) if ref_pins.RECORD else impl
        else:
            _mods[key] = ref_pins.stand_in(kind)
    return _mods[key]


def module(pinned=False):
    """The compiled reference raycaster extension; with ``pinned``, the recorded stand-in where it is not built."""
    return _module("raycast", RAYCAST_SO, pinned)


def depth_module(pinned=False):
    """The compiled reference depth_utils extension (oracle/build_ref.py::build_depth); ``pinned`` as for module()."""
    return _module("depth", DEPTH_SO, pinned)


def ref_depth2normals(depth, intrinsics, filter_helper, camspace, normals, max_num_fill_iters=40, pinned=False):
    """Depth2Normals.forward of the reference, statement by statement (depth_utils.py:84-100), on its native entry points."""
    m = depth_module(pinned)
    m.bilateral_filter_floatmap(filter_helper, depth, 2.0, 0.1)
    if max_num_fill_iters > 0:
        invalid = bool((depth == 0).any())
        for _ in range(max_num_fill_iters // 2):
            if not invalid:
                break
            m.median_fill_depthmap(depth, filter_helper)      # median_fill_depthmap(filt, img, 2), depth_utils.py:55-59
            m.median_fill_depthmap(filter_helper, depth)
            invalid = bool((depth == 0).any())
        if invalid:
            return None
    m.convert_depth_to_cameraspace(camspace, depth, intrinsics, 0.0, 0.0)
    m.compute_normals(normals, camspace)
    return normals.permute(0, 3, 1, 2).contiguous()


class RefRaycaster:
    def __init__(self, batch_size, dims3d, width, height, depth_min, depth_max, thresh, inc, max_locs, max_pix=64,
                 device="cuda", pinned=False):
        self.module = module(pinned)
        self.args = (batch_size, dims3d, width, height, depth_min, depth_max, thresh, inc)
        z = lambda *s, **k: torch.zeros(*s, device=device, **k)
        self.image_depth = z(batch_size, height, width)
        self.image_normal = z(batch_size, height, width, 3)
        self.image_color = z(batch_size, height, width, 3)
        self.image_semantic = z(batch_size, height, width, 14)
        self.mapping3dto2d = z(batch_size * max_locs, max_pix, dtype=torch.int)
        self.mapping3dto2d_num = z(batch_size * max_locs, dtype=torch.int)
        self.sparse_mapping = z(batch_size, dims3d[0], dims3d[1], dims3d[2], dtype=torch.int)
        self.d_color = z(batch_size * max_locs, 3)
        self.d_normal = z(batch_size * max_locs, 3)
        self.d_depth = z(batch_size * max_locs, 1)
        self.d_semantic = z(batch_size * max_locs, 14)

    def forward(self, locs, sdf, color, normal, semantic, view, intr):
        b, dims3d, w, h, dmin, dmax, thresh, inc = self.args
        m = self.module
        m.construct_dense_sparse_mapping(locs, self.sparse_mapping)
        opts = torch.FloatTensor([w, h, dmin, dmax, thresh, inc, dims3d[2], dims3d[1], dims3d[0]])
        m.forward(self.sparse_mapping, locs, sdf, color, normal, semantic, view, self.image_color, self.image_depth,
                  self.image_normal, self.image_semantic, self.mapping3dto2d, self.mapping3dto2d_num, intr, opts)
        self.n = locs.shape[0]
        return self.image_color, self.image_depth, self.image_normal, self.image_semantic

    def backward(self, g_color, g_depth, g_normal, g_semantic):
        b, dims3d = self.args[0], self.args[1]
        dims = torch.IntTensor([b, dims3d[2], dims3d[1], dims3d[0], self.n])
        self.module.backward(g_color.contiguous(), g_depth.contiguous(), g_normal.contiguous(), g_semantic.contiguous(),
                             self.sparse_mapping, self.mapping3dto2d, self.mapping3dto2d_num, dims, self.d_color,
                             self.d_depth, self.d_normal, self.d_semantic)
        n = self.n
        return self.d_color[:n], self.d_depth[:n], self.d_normal[:n], self.d_semantic[:n]
