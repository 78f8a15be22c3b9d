"""Label render without a GPU: spsg_raycast_labels is declared and exported, its ctypes mirror matches the header, its
argument checks return before anything is enqueued, and no label-mode kernel uses floating-point atomics."""
import ctypes
import os
import re

import pytest

from spsg_b200 import _native as N
from tests.test_deterministic_cpu import _FLOAT_ATOMIC, _sass_functions

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "spsg_raycast.h")
FAKE = 1 << 20  # never dereferenced: every check below fails before the device is touched
INVALID, TOO_SMALL = 1, 3  # SPSG_ERR_INVALID_ARGUMENT, SPSG_ERR_WORKSPACE_TOO_SMALL


def _params(c=0, n=1000, flags=0, b=2, f=3):
    return N.make_params(160, 128, 0.1, 6.0, 1.0, 0.9, 64, 64, 128, b, f, 64, n, flags, c)


def _call(p, ws_bytes=None, sparse=FAKE, locs=FAKE, sdf=FAKE, labels=FAKE, view=FAKE, intr=FAKE, out=FAKE, hist=None,
          ws=FAKE):
    if ws_bytes is None:
        ws_bytes = N.lib.spsg_workspace_bytes(ctypes.byref(_params()))
    return N.lib.spsg_raycast_labels(ctypes.byref(p) if p is not None else None, sparse, locs, sdf, labels, view, intr,
                                     out, hist, ws, ws_bytes, None)


def test_declared_exported_and_mirrored():
    with open(HEADER) as fh:
        src = fh.read()
    m = re.search(r"SPSG_API int spsg_raycast_labels\((.*?)\);", src, re.S)
    assert m, "spsg_raycast_labels is not declared"
    args = [a.strip() for a in m.group(1).split(",")]
    assert [a.split()[-1].lstrip("*") for a in args] == [
        "p", "sparse_mapping", "locs", "vals_sdf", "voxel_labels", "view_matrix", "intrinsics", "image_label", "hist",
        "workspace", "workspace_bytes", "stream"]
    assert "uint8_t *voxel_labels" in m.group(1) and "uint8_t *image_label" in m.group(1) and "int64_t *hist" in m.group(1)
    assert "spsg_raycast_labels" in N.EXPORTS and hasattr(N.lib, "spsg_raycast_labels")
    f = N.lib.spsg_raycast_labels
    assert f.restype == ctypes.c_int and len(f.argtypes) == len(args)
    assert f.argtypes[0] == ctypes.POINTER(N.Params) and f.argtypes[-2] == ctypes.c_size_t


@pytest.mark.parametrize("c", [65, 100, 1 << 31])
def test_out_of_range_c_is_rejected(c):
    assert _call(_params(c)) == INVALID
    assert b"semantic_channels" in N.lib.spsg_last_error()


def test_null_pointers_are_rejected():
    assert _call(None) == INVALID
    for kw in ("sparse", "view", "intr", "out", "locs", "sdf", "labels"):
        assert _call(_params(), **{kw: None}) == INVALID, kw
        assert b"NULL" in N.lib.spsg_last_error(), kw
    # without voxels, the voxel tensors may be NULL (the workspace check fails next: nothing reaches the device)
    assert _call(_params(n=0), locs=None, sdf=None, labels=None, ws_bytes=16) == TOO_SMALL


def test_misaligned_pointers_are_rejected():
    assert _call(_params(), locs=FAKE + 8) == INVALID
    assert _call(_params(flags=N.SPSG_FLAG_PACKED_LOCS), locs=FAKE + 2) == INVALID
    assert _call(_params(), view=FAKE + 4) == INVALID
    assert _call(_params(), hist=FAKE + 4) == INVALID


def test_short_workspace_is_rejected():
    need = N.lib.spsg_workspace_bytes(ctypes.byref(_params()))
    assert _call(_params(), ws_bytes=need - 1) == TOO_SMALL
    assert _call(_params(), ws=None) == TOO_SMALL
    assert _call(_params(), ws=FAKE + 128) == INVALID  # 256-byte alignment


@pytest.mark.parametrize("flags", [N.SPSG_FLAG_DETERMINISTIC, N.SPSG_FLAG_ALL_PIXELS,
                                   N.SPSG_FLAG_DETERMINISTIC | N.SPSG_FLAG_ALL_PIXELS | N.SPSG_FLAG_VIEW_NORMALS])
def test_needs_no_more_than_the_plain_workspace(flags):
    """Flags that grow spsg_workspace_bytes concern tables and losses: the label render ignores them and needs only the
    workspace of the call without them (it is refused one byte below that, not below the flagged size)."""
    plain = N.lib.spsg_workspace_bytes(ctypes.byref(_params()))
    assert N.lib.spsg_workspace_bytes(ctypes.byref(_params(flags=flags))) > plain
    assert _call(_params(flags=flags), ws_bytes=plain - 1) == TOO_SMALL


def test_label_kernels_use_no_float_atomics():
    funcs = _sass_functions()
    label = {k: v for k, v in funcs.items() if re.search(r"raycast_forward_kernelILb0ELb[01]ELi\d+ELb0ELb0ELb1E", k)}
    assert len(label) == 4, sorted(label)  # maps in shared memory or through L1, 24 or 28 warps
    for name, lines in label.items():
        bad = [x for x in lines if _FLOAT_ATOMIC.search(x)]
        assert not bad, (name, bad[:3])
        assert any(re.search(r"\bATOMS\.", x) for x in lines), "%s: no shared-memory histogram atomics" % name
