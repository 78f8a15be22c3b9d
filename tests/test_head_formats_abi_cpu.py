"""The bfloat16 compaction and strided gather / scatter entry points: exported, and their argument validation runs before
anything touches the device, so it is checked here without a GPU (the pointers are never dereferenced)."""
import ctypes

SPSG_ERR_INVALID_ARGUMENT = 1  # include/spsg_raycast.h

NEW = ("spsg_sparsify_count_bf16", "spsg_sparsify_locs_bf16", "spsg_sparsify_locs_indexed_bf16",
       "spsg_dense_gather_strided", "spsg_dense_scatter_strided")


def test_new_symbols_are_exported():
    from spsg_b200 import _native as N
    for name in NEW:
        assert name in N.EXPORTS
        assert hasattr(N.lib, name)


def _head(N, dtype=0, channels=3, strides=None, extent=None, dense=0x10000, sparse=0x20000):
    B, C, D = 2, channels, (4, 5, 6)
    if strides is None:  # NDHWC-contiguous
        strides = (D[0] * D[1] * D[2] * C, 1, D[1] * D[2] * C, D[2] * C, C)
    if extent is None:
        extent = B * C * D[0] * D[1] * D[2]
    return N.DenseHead(dense, sparse, (ctypes.c_int64 * 5)(*strides), extent, channels, dtype)


def _call(N, fn, heads, num_locs=0, locs=0x30000, grid=(2, 4, 5, 6)):
    arr = (N.DenseHead * len(heads))(*heads)
    return fn(arr, len(heads), locs, num_locs, *grid, None)


def test_strided_gather_scatter_validate_their_arguments():
    from spsg_b200 import _native as N
    for fn in (N.lib.spsg_dense_gather_strided, N.lib.spsg_dense_scatter_strided):
        bad = [
            [_head(N, dtype=2)],                                    # unknown dtype
            [_head(N, dtype=-1)],
            [_head(N, channels=0)],                                 # non-positive channels
            [_head(N, dense=None)],                                 # NULL dense
            [_head(N, extent=2 * 3 * 4 * 5 * 6 - 1)],               # last element beyond the extent
            [_head(N, strides=(360, 1, 90, 18, -3))],               # negative stride
            [_head(N, dtype=1, dense=0x10001)],                     # bf16 head not 2-byte aligned
            [_head(N, dense=0x10002)],                              # f32 head not 4-byte aligned
            [_head(N)] * 5,                                         # more than 4 heads
        ]
        for heads in bad:
            assert _call(N, fn, heads) == SPSG_ERR_INVALID_ARGUMENT, heads[0].dtype
        assert _call(N, fn, [_head(N, sparse=None)], num_locs=7) == SPSG_ERR_INVALID_ARGUMENT   # NULL sparse
        assert _call(N, fn, [_head(N)], num_locs=7, locs=None) == SPSG_ERR_INVALID_ARGUMENT     # NULL locs
        assert _call(N, fn, [_head(N)], grid=(0, 4, 5, 6)) == SPSG_ERR_INVALID_ARGUMENT         # non-positive size
        assert _call(N, fn, [_head(N)], grid=(2, 4, -5, 6)) == SPSG_ERR_INVALID_ARGUMENT
        # well-formed, no heads: nothing to do
        assert _call(N, fn, []) == 0
    # a gather reads a channel slice in place (strides of the 19-channel parent), a scatter needs a packed target
    sl = _head(N, channels=3, strides=(4 * 5 * 6 * 19, 1, 5 * 6 * 19, 6 * 19, 19), extent=2 * 19 * 4 * 5 * 6 - 5)
    assert _call(N, N.lib.spsg_dense_scatter_strided, [sl]) == SPSG_ERR_INVALID_ARGUMENT
    assert b"packed" in N.lib.spsg_last_error()
    assert _call(N, N.lib.spsg_dense_gather_strided, [sl]) == 0           # no rows: validated, nothing launched


def test_bf16_compaction_validates_its_arguments():
    from spsg_b200 import _native as N
    scratch = 0x100000
    nbytes = N.lib.spsg_sparsify_scratch_bytes(1000)
    assert N.lib.spsg_sparsify_count_bf16(None, None, 1000, 3.0, scratch, nbytes, 0x200000, None) == \
        SPSG_ERR_INVALID_ARGUMENT
    assert N.lib.spsg_sparsify_count_bf16(0x10008, None, 1000, 3.0, scratch, nbytes, 0x200000, None) == \
        SPSG_ERR_INVALID_ARGUMENT                                                # sdf not 16-byte aligned
    assert N.lib.spsg_sparsify_count_bf16(0x10000, None, 0, 3.0, scratch, nbytes, 0x200000, None) == \
        SPSG_ERR_INVALID_ARGUMENT                                                # no cells
    assert N.lib.spsg_sparsify_locs_bf16(0x10000, None, 0, 10, 10, 10, 3.0, scratch, 0x300000, 5, None) == \
        SPSG_ERR_INVALID_ARGUMENT                                                # non-positive grid
    assert N.lib.spsg_sparsify_locs_bf16(None, None, 1, 10, 10, 10, 3.0, scratch, 0x300000, 5, None) == \
        SPSG_ERR_INVALID_ARGUMENT                                                # NULL sdf
    assert N.lib.spsg_sparsify_locs_indexed_bf16(0x10000, None, 1, 10, 10, 10, 3.0, scratch, 0x300000, 5, None,
                                                 0x400000, None) == SPSG_ERR_INVALID_ARGUMENT   # NULL index
    assert N.lib.spsg_sparsify_locs_bf16(0x10000, None, 1, 10, 10, 10, 3.0, scratch, 0x300000, 0, None) == 0
