"""The per-view normals entry points and SPSG_FLAG_VIEW_NORMALS: exported, bound, and their argument checks run before
anything touches the device, so they are checked here without a GPU (the pointers are never dereferenced)."""
import ctypes

SPSG_ERR_INVALID_ARGUMENT = 1  # include/spsg_raycast.h
FAKE = 0x2000  # any non-NULL, 256-byte aligned address


def _forward(N, views, transform):
    return N.lib.spsg_normals_forward_views(FAKE, 10, FAKE, transform, views, FAKE, 2, 8, 8, 8, FAKE, None)


def _backward(N, views, transform):
    return N.lib.spsg_normals_backward_views(FAKE, 10, FAKE, transform, views, FAKE, 2, 8, 8, 8, FAKE, FAKE, FAKE, None)


def test_entry_points_are_exported_and_the_flag_is_bit_9():
    from spsg_b200 import _native as N
    lib = ctypes.CDLL(N.LIB_PATH)
    for name in ("spsg_normals_forward_views", "spsg_normals_backward_views"):
        assert name in N.EXPORTS
        assert hasattr(lib, name)
    assert N.SPSG_FLAG_VIEW_NORMALS == 1 << 9


def test_views_per_chunk_must_be_positive():
    from spsg_b200 import _native as N
    for views in (0, -1, -5):
        for call in (_forward, _backward):
            assert call(N, views, FAKE) == SPSG_ERR_INVALID_ARGUMENT
            assert b"views_per_chunk" in N.lib.spsg_last_error()


def test_several_views_need_a_transform():
    from spsg_b200 import _native as N
    for views in (2, 3, 5):
        for call in (_forward, _backward):
            assert call(N, views, None) == SPSG_ERR_INVALID_ARGUMENT
            assert b"transform" in N.lib.spsg_last_error()


def test_bad_sizes_are_rejected_in_the_per_view_path():
    from spsg_b200 import _native as N
    # num_chunks 0 with F > 1 reaches the shared size checks, still before any launch
    assert N.lib.spsg_normals_forward_views(FAKE, 10, FAKE, FAKE, 3, FAKE, 0, 8, 8, 8, FAKE, None) == \
        SPSG_ERR_INVALID_ARGUMENT
    assert N.lib.spsg_normals_backward_views(FAKE, 10, FAKE, FAKE, 3, None, 2, 8, 8, 8, FAKE, FAKE, FAKE, None) == \
        SPSG_ERR_INVALID_ARGUMENT
