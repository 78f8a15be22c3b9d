"""All-pixels mode (SPSG_FLAG_ALL_PIXELS) without a GPU: the flag's value, the workspace it adds, the NULL-table rule,
the SASS of the kernels its deterministic calls launch, and the uncapped-gather emulation of tests/fuzz_all_pixels.py
against fuzz_deterministic.exact_gather."""
import ctypes
import os
import re

import numpy as np
import pytest

from spsg_b200 import _native as N

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _params(w, h, b, f, p, n, flags):
    return N.make_params(w, h, 0.1, 6.0, 1.0, 0.9, 64, 64, 128, b, f, p, n, flags)


def test_flag_value_matches_the_header():
    with open(os.path.join(ROOT, "include", "spsg_raycast.h")) as fh:
        m = re.search(r"SPSG_FLAG_ALL_PIXELS\s*=\s*1u\s*<<\s*(\d+)", fh.read())
    assert m and N.SPSG_FLAG_ALL_PIXELS == 1 << int(m.group(1)) == 1 << 11


def _a(b):
    return (b + 255) // 256 * 256


@pytest.mark.parametrize("w,h,b,f,n", [(320, 256, 8, 1, 640000 * 8), (160, 128, 3, 2, 123457), (33, 17, 1, 4, 0)])
def test_workspace_grows_only_with_the_flag(w, h, b, f, n):
    for extra in (0, N.SPSG_FLAG_DETERMINISTIC, N.SPSG_FLAG_VIEW_NORMALS | N.SPSG_FLAG_DETERMINISTIC_GRADS):
        base = N.lib.spsg_workspace_bytes(ctypes.byref(_params(w, h, b, f, 64, n, extra)))
        for p in (64, 0, 7):  # max_pixels_per_voxel is ignored with the flag
            got = N.lib.spsg_workspace_bytes(ctypes.byref(_params(w, h, b, f, p, n, extra | N.SPSG_FLAG_ALL_PIXELS)))
            px = b * f * w * h
            want = base + 256 + _a(4 * f * n) + _a(4 * px)
            if extra & N.SPSG_FLAG_DETERMINISTIC:
                want += _a(4 * (px // 65 + 1))
            assert got == want, (extra, p, got, want)


def test_null_table_only_with_the_flag():
    fake = 1 << 20  # never dereferenced: validation returns before anything is enqueued (1 = invalid argument, 3 = workspace
    # too small, 0 = ok)
    args14 = [fake] * 12 + [None, fake]  # mapping3dto2d NULL
    small = 256
    p = _params(80, 64, 1, 1, 64, 100, 0)
    assert N.lib.spsg_raycast_forward(ctypes.byref(p), *args14, fake, small, None) == 1
    p.flags = N.SPSG_FLAG_ALL_PIXELS
    p.max_pixels_per_voxel = 0
    assert N.lib.spsg_raycast_forward(ctypes.byref(p), *args14, fake, small, None) == 3
    p.max_pixels_per_voxel = 0
    p.flags = 0
    assert N.lib.spsg_raycast_forward(ctypes.byref(p), *([fake] * 14), fake, small, None) == 1
    # backward entry points: num_locs = 0 returns after validation
    q = _params(80, 64, 1, 1, 64, 0, 0)
    bargs = [fake] * 5 + [None, fake] + [fake] * 4
    assert N.lib.spsg_raycast_backward(ctypes.byref(q), *bargs, fake, small, None) == 1
    q.flags = N.SPSG_FLAG_ALL_PIXELS
    assert N.lib.spsg_raycast_backward(ctypes.byref(q), *bargs, fake, small, None) == 0
    tg = N.LossTargets(fake, None, None, None, None, 0.02, 1.0, 1.0, 1.0)
    up = N.UpstreamGrads(fake, None, None, None)
    for flags, rc in ((0, 1), (N.SPSG_FLAG_ALL_PIXELS, 0)):
        q.flags = flags
        assert N.lib.spsg_raycast_backward_loss(ctypes.byref(q), fake, fake, fake, ctypes.byref(tg), fake, None, fake, None,
                                                fake, fake, fake, fake, fake, fake, small, None) == rc
        assert N.lib.spsg_raycast_backward_loss_upstream(ctypes.byref(q), fake, fake, fake, ctypes.byref(tg), fake, None,
                                                         ctypes.byref(up), fake, None, fake, fake, fake, fake, fake, fake,
                                                         small, None) == rc


def test_deterministic_kernels_have_no_float_atomics():
    from tests.test_deterministic_cpu import _FLOAT_ATOMIC, _sass_functions
    funcs = _sass_functions()
    seen = set()
    pats = (r"seg_alloc_kernel", r"seg_scatter_kernel", r"seg_sort_warp_kernel", r"seg_sort_long_kernel",
            r"backward_gather_kernelILb[01]ELb[01]ELi[02]ELb[01]ELb1E")
    for name, lines in funcs.items():
        for pat in pats:
            if re.search(pat, name):
                seen.add(pat)
                bad = [ln.strip() for ln in lines if _FLOAT_ATOMIC.search(ln)]
                assert not bad, "%s: %s" % (name, bad[:3])
    assert seen == set(pats)
    # the float-atomic variant of the segment gather (several views, default mode) does have them
    assert any(_FLOAT_ATOMIC.search(ln) for name, lines in funcs.items()
               if re.search(r"backward_gather_kernelILb0ELb0ELi1ELb0ELb1E", name) for ln in lines)


def test_uncapped_emulation_equals_exact_gather():
    from tests import fuzz_all_pixels as A
    from tests import fuzz_deterministic as D
    rng = np.random.default_rng(0)
    for F, n, images_per_chunk, P in ((1, 40, 1, 300), (3, 25, 3, 500)):
        chunks = 2
        chunk = np.repeat(np.arange(chunks), n // chunks + 1)[:n]
        vox = np.full((chunks * F, P), -1, np.int64)
        for img in range(chunks * F):
            mine = np.nonzero(chunk == img // F)[0]
            hit = rng.random(P) < 0.8
            vox[img, hit] = rng.choice(mine[:3], hit.sum())  # few voxels: long rows
        c = A.all_tables(vox, chunk, F)
        G = rng.standard_normal((chunks * F * P, 21)).astype(np.float32) * np.float32(2.0) ** rng.integers(-20, 20, (1, 21))
        want = D.exact_gather(c, G)
        got = A.exact_gather(c, G)[0]
        assert np.array_equal(D.bits(got), D.bits(want))
