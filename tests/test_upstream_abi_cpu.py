"""Argument validation of spsg_raycast_backward_loss_upstream: it runs before anything touches the device, so it is
checked here without a GPU (the pointers are never dereferenced)."""
import ctypes

SPSG_ERR_INVALID_ARGUMENT = 1  # include/spsg_raycast.h


def _call(N, p, image_color=0x1000, upstream=None):
    fake = 0x2000  # any non-NULL, 256-byte aligned address
    tg = N.LossTargets(None, None, None, None, None, 0.02, 1.0, 1.0, 1.0)
    return N.lib.spsg_raycast_backward_loss_upstream(
        ctypes.byref(p), image_color, fake, fake, ctypes.byref(tg), fake, None,
        None if upstream is None else ctypes.byref(upstream), fake, fake, fake, fake, fake, fake, fake, fake, 1 << 20,
        None)


def test_upstream_entry_point_validates_its_arguments():
    from spsg_b200 import _native as N
    p = N.make_params(320, 256, 5, 300, 45.45, 0.9, 64, 64, 128, 1, 1, 64, 0)
    # misaligned grad_semantic
    bad = N.UpstreamGrads(None, None, None, 0x3004)
    assert _call(N, p, upstream=bad) == SPSG_ERR_INVALID_ARGUMENT
    assert b"grad_semantic" in N.lib.spsg_last_error()
    # NULL mandatory pointer, with and without upstream planes
    up = N.UpstreamGrads(0x3000, None, 0x4000, 0x5008)
    for u in (up, None):
        assert _call(N, p, image_color=None, upstream=u) == SPSG_ERR_INVALID_ARGUMENT
        assert b"NULL" in N.lib.spsg_last_error()
    # well-formed arguments and no voxels: nothing to launch
    assert _call(N, p, upstream=up) == 0
    assert _call(N, p, upstream=N.UpstreamGrads(None, None, None, None)) == 0

