"""Eval render without a GPU: spsg_raycast_eval and its scratch size are declared and exported, the ctypes mirror matches
the header, bad arguments are refused before anything is enqueued, spsg_workspace_bytes does not change, and no eval
kernel uses floating-point atomics."""
import ctypes
import os
import re

import pytest

from spsg_b200 import _native as N
from tests.test_deterministic_cpu import _FLOAT_ATOMIC, _sass_functions

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "spsg_raycast.h")
FAKE = 1 << 20  # never dereferenced: every check below fails before the device is touched
INVALID, TOO_SMALL = 1, 3


def _params(c=0, n=1000, flags=0, b=2, f=3):
    return N.make_params(160, 128, 0.1, 6.0, 1.0, 0.9, 64, 64, 128, b, f, 64, n, flags, c)


def _call(p, targets=True, label=True, loss_out=FAKE, conf=None, scratch=FAKE, scratch_bytes=None, ws=FAKE, ws_bytes=None,
          **ptrs):
    if ws_bytes is None:
        ws_bytes = N.lib.spsg_workspace_bytes(ctypes.byref(_params()))
    if scratch_bytes is None:
        scratch_bytes = N.lib.spsg_raycast_eval_scratch_bytes(ctypes.byref(_params()))
    tg = N.LossTargets(FAKE, FAKE, None, FAKE if label else None, None, 0.02, 1.0, 1.0, 1.0)
    a = [ptrs.get(k, FAKE) for k in ("sparse", "locs", "sdf", "color", "sem", "pred", "view", "intr")]
    return N.lib.spsg_raycast_eval(ctypes.byref(p) if p is not None else None, *a, ctypes.byref(tg) if targets else None,
                                   loss_out, None, conf, scratch, scratch_bytes, ws, ws_bytes, None)


def test_declared_exported_and_mirrored():
    with open(HEADER) as fh:
        src = fh.read()
    m = re.search(r"SPSG_API int spsg_raycast_eval\((.*?)\);", src, re.S)
    assert m, "spsg_raycast_eval is not declared"
    args = [a.strip() for a in m.group(1).split(",")]
    assert [a.split()[-1].lstrip("*") for a in args] == [
        "p", "sparse_mapping", "locs", "vals_sdf", "vals_color", "vals_semantic", "pred_labels", "view_matrix", "intrinsics",
        "t", "loss_out", "image_label", "confusion", "scratch", "scratch_bytes", "workspace", "workspace_bytes", "stream"]
    assert "uint64_t *confusion" in m.group(1) and "const spsg_loss_targets *t" in m.group(1)
    assert re.search(r"SPSG_API size_t spsg_raycast_eval_scratch_bytes\(const spsg_raycast_params \*p\);", src)
    for name in ("spsg_raycast_eval", "spsg_raycast_eval_scratch_bytes"):
        assert name in N.EXPORTS and hasattr(N.lib, name)
    f = N.lib.spsg_raycast_eval
    assert f.restype == ctypes.c_int and len(f.argtypes) == len(args)
    assert f.argtypes[0] == ctypes.POINTER(N.Params) and f.argtypes[9] == ctypes.POINTER(N.LossTargets)
    assert f.argtypes[14] == ctypes.c_size_t and f.argtypes[16] == ctypes.c_size_t
    assert N.lib.spsg_raycast_eval_scratch_bytes.restype == ctypes.c_size_t


def test_scratch_bytes():
    # 8 floats per 8x4 warp tile: 160x128 -> 20 x 32 tiles (in 16x8 blocks of four) per image, 6 images
    tiles = 10 * 16 * 4 * 6
    got = N.lib.spsg_raycast_eval_scratch_bytes(ctypes.byref(_params()))
    assert tiles * 32 <= got <= tiles * 32 + 4096 + 256 + 512 + 256
    assert N.lib.spsg_raycast_eval_scratch_bytes(ctypes.byref(_params(c=65))) == 0
    # independent of C and of every flag
    for p in (_params(c=64), _params(flags=N.SPSG_FLAG_DETERMINISTIC | N.SPSG_FLAG_ALL_PIXELS)):
        assert N.lib.spsg_raycast_eval_scratch_bytes(ctypes.byref(p)) == got


@pytest.mark.parametrize("c", [65, 100, 1 << 31])
def test_out_of_range_c_is_rejected(c):
    assert _call(_params(c)) == INVALID
    assert b"semantic_channels" in N.lib.spsg_last_error()


def test_null_and_missing_arguments_are_rejected():
    assert _call(None) == INVALID
    assert _call(_params(), targets=False) == INVALID
    assert _call(_params(), loss_out=None) == INVALID
    assert _call(_params(), label=False, conf=FAKE) == INVALID and b"target labels" in N.lib.spsg_last_error()
    for kw in ("sparse", "view", "intr", "locs", "sdf", "pred", "color", "sem"):
        assert _call(_params(), **{kw: None}) == INVALID, kw
        assert b"NULL" in N.lib.spsg_last_error(), kw
    # colour / logits may be NULL when their term is off; without voxels every voxel tensor may be NULL
    assert _call(_params(), label=False, sem=None, ws_bytes=16) == TOO_SMALL
    assert _call(_params(n=0), locs=None, sdf=None, color=None, sem=None, pred=None, ws_bytes=16) == TOO_SMALL


def test_misaligned_pointers_are_rejected():
    assert _call(_params(), locs=FAKE + 8) == INVALID
    assert _call(_params(flags=N.SPSG_FLAG_PACKED_LOCS), locs=FAKE + 2) == INVALID
    assert _call(_params(), view=FAKE + 4) == INVALID
    assert _call(_params(), conf=FAKE + 4) == INVALID
    assert _call(_params(), scratch=FAKE + 128) == INVALID


def test_short_scratch_and_workspace_are_rejected():
    need = N.lib.spsg_raycast_eval_scratch_bytes(ctypes.byref(_params()))
    assert _call(_params(), scratch_bytes=need - 1) == TOO_SMALL
    assert _call(_params(), scratch=None) == TOO_SMALL
    plain = N.lib.spsg_workspace_bytes(ctypes.byref(_params()))
    assert _call(_params(), ws_bytes=plain - 1) == TOO_SMALL
    assert _call(_params(), ws=None) == TOO_SMALL
    assert _call(_params(), ws=FAKE + 128) == INVALID
    # flags that grow spsg_workspace_bytes are ignored: the plain size is enough
    flags = N.SPSG_FLAG_DETERMINISTIC | N.SPSG_FLAG_ALL_PIXELS
    assert N.lib.spsg_workspace_bytes(ctypes.byref(_params(flags=flags))) > plain
    assert _call(_params(flags=flags), ws_bytes=plain - 1) == TOO_SMALL


# spsg_workspace_bytes of the library before the eval render existed, for these parameter sets
_WORKSPACE_BYTES = {(0, 1, 1, 0): 2331392, (0, 2, 3, 1000): 5009664, (0, 8, 5, 123457): 26177280,
                    (1024, 1, 1, 0): 2331904, (1024, 2, 3, 1000): 5011712, (1024, 8, 5, 123457): 26190080,
                    (2048, 1, 1, 0): 2413568, (2048, 2, 3, 1000): 5513472, (2048, 8, 5, 123457): 31923712}


def test_workspace_bytes_unchanged():
    """The eval render adds nothing to spsg_workspace_bytes, for any C, mode, batch or voxel count."""
    for (flags, b, f, n), want in _WORKSPACE_BYTES.items():
        for c in (0, 1, 14, 64):
            assert N.lib.spsg_workspace_bytes(ctypes.byref(_params(c=c, n=n, flags=flags, b=b, f=f))) == want, (c, flags, b, f, n)


def test_eval_kernels_use_no_float_atomics():
    funcs = _sass_functions()
    ev = {k: v for k, v in funcs.items() if re.search(r"raycast_forward_kernelILb0ELb[01]ELi\d+ELb0ELb0ELb0ELb1E", k)}
    assert len(ev) == 4, sorted(ev)  # maps in shared memory or through L1, 24 or 28 warps
    total = {k: v for k, v in funcs.items() if "eval_loss_sum_kernel" in k}
    assert len(total) == 1
    for name, lines in list(ev.items()) + list(total.items()):
        bad = [x for x in lines if _FLOAT_ATOMIC.search(x)]
        assert not bad, (name, bad[:3])
    for name, lines in ev.items():
        assert any(re.search(r"\bATOMS\.", x) for x in lines), "%s: no shared-memory confusion atomics" % name
