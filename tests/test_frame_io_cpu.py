"""frame_io.load_frames (drop-in for data_util.load_frames, data_util.py:862-902) against the reference's own function on
small synthetic frame files.  The reference decodes with `imageio.imread`, which this image lacks; for these formats
imageio itself decodes with Pillow, so a three-line stand-in (`imread = numpy.array(PIL.Image.open(f))`) is registered
for it -- everything after decoding (resize, crop, scaling, intrinsic adjustment, batching) is the reference's code."""
import hashlib
import os
import sys
import types

import numpy as np
import pytest
import torch
from PIL import Image


def _write_scene(root, scene, frame_ids, size_wh, rng):
    for sub in ("depth", "color", "camera"):
        os.makedirs(os.path.join(root, scene, sub), exist_ok=True)
    w, h = size_wh
    for f in frame_ids:
        depth = rng.integers(0, 6000, size=(h, w)).astype(np.uint16)
        depth[rng.random((h, w)) < 0.1] = 0
        Image.fromarray(depth).save(os.path.join(root, scene, "depth", "%d.png" % f))
        color = rng.integers(0, 256, size=(h, w, 3)).astype(np.uint8)
        Image.fromarray(color).save(os.path.join(root, scene, "color", "%d.jpg" % f), quality=95)
        pose = np.eye(4) + rng.standard_normal((4, 4)) * 0.1
        intr = np.array([[1075.0 + f, 0, w / 2 - 0.5, 0], [0, 1076.0, h / 2 - 0.5, 0], [0, 0, 1, 0], [0, 0, 0, 1]])
        with open(os.path.join(root, scene, "camera", "%d.txt" % f), "w") as fh:
            for row in list(pose) + list(intr):
                fh.write(" ".join("%.6f" % v for v in row) + "\n")


GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "frame_io_ref.npz")
CASES = [((64, 48), (40, 32)), ((80, 64), (80, 64)), ((96, 40), (32, 24))]


def _golden_key(src_wh, dst_wh):
    return "%dx%d_%dx%d" % (src_wh + dst_wh)


def digest(t):
    """SHA-256 of a tensor's dtype, shape and bytes: equal digests <=> torch.equal (the stored form of the images)."""
    t = t.contiguous()
    return hashlib.sha256(("%s%s" % (t.dtype, tuple(t.shape))).encode() + t.view(torch.uint8).numpy().tobytes()).hexdigest()


def _stored_reference(src_wh, dst_wh):
    """What the reference's data_util.load_frames returned on this case (tests/golden/make_golden_frame_io.py): the
    images as digests, poses, intrinsics and frame ids as values."""
    g = np.load(GOLDEN)
    k = _golden_key(src_wh, dst_wh)
    t = lambda name: torch.from_numpy(g[k + name])
    d = lambda name: str(g[k + name])
    want = (d("_depth"), d("_color"), t("_pose"), t("_intr"), [list(r) for r in g[k + "_frameids"]])
    want_self = (d("_self_depth"), None, None, t("_self_intr"))
    return want, want_self


def _equal(got, want):
    return digest(got) == want if isinstance(want, str) else got.shape == want.shape and torch.equal(got, want)


def _reference_data_util():
    from baseline import ref_loader
    if not ref_loader.available():
        return None
    shim = types.ModuleType("imageio")
    shim.imread = lambda f: np.array(Image.open(f))
    sys.modules["imageio"] = shim
    du = ref_loader.load_module("data_util")
    du.imageio = shim
    return du


def reference_outputs(du, tmp_path, src_wh, dst_wh):
    """The case's inputs written under tmp_path; (frame_io.load_frames argument tuple, the reference's outputs on it,
    the same with 'self' frame ids and depth only).  `du` is the reference's data_util, or None for the stored
    outputs."""
    rng = np.random.default_rng(5)
    names = ["sceneA_room0__inc__3", "sceneB_room2__inc__1"]
    ids = {"sceneA": [3, 7, 9], "sceneB": [1, 2, 4]}
    for scene, fr in ids.items():
        _write_scene(str(tmp_path / "images"), scene, fr, src_wh, rng)
    os.makedirs(tmp_path / "frames")
    for name in names:
        with open(tmp_path / "frames" / (name.replace("__inc__", "__cmp__") + ".txt"), "w") as fh:
            fh.write("\n".join(str(i) for i in ids[name.split("_room")[0]]) + "\n")
    args = (names, None, str(tmp_path / "frames"), str(tmp_path / "images"), False, list(dst_wh), list(dst_wh), None, True, True)
    args_self = (names, None, "self", str(tmp_path / "images"), False, list(dst_wh), list(dst_wh), None, True, False)
    if du is None:
        want, want_self = _stored_reference(src_wh, dst_wh)
    else:
        want, want_self = du.load_frames(*args, max_num_frames=2), du.load_frames(*args_self)
    return args, args_self, want, want_self


@pytest.mark.parametrize("src_wh,dst_wh", CASES)
def test_load_frames_matches_reference(tmp_path, src_wh, dst_wh):
    """Against the reference's function where baseline/_ref is installed, else against its stored outputs."""
    from spsg_b200 import frame_io
    args, args_self, want, want_self = reference_outputs(_reference_data_util(), tmp_path, src_wh, dst_wh)
    for workers in (0, 4):
        got = frame_io.load_frames(*args, max_num_frames=2, num_workers=workers)
        for a, b in zip(got[:4], want[:4]):
            assert _equal(a, b)
        assert [list(f) for f in got[4]] == [list(f) for f in want[4]]
    # 'self' frame ids, depth only, too few frames
    got = frame_io.load_frames(*args_self)
    assert got[1] is None and want_self[1] is None and _equal(got[0], want_self[0]) and _equal(got[3], want_self[3])
    assert frame_io.load_frames(*args, max_num_frames=5) == (None, None, None, None, None)
