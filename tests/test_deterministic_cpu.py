"""Deterministic mode without a GPU: the flag's ABI, the workspace it needs, argument validation, and the SASS of the
kernels a deterministic call launches (no floating-point atomics)."""
import ctypes
import os
import re
import shutil
import subprocess

import pytest

from spsg_b200 import _native as N


def _params(w, h, dx, dy, dz, b, f, p, n, flags):
    return N.make_params(w, h, 0.1, 6.0, 1.0, 0.9, dx, dy, dz, b, f, p, n, flags)


# (params, spsg_workspace_bytes before the flag existed)
_SIZES = [((320, 256, 64, 64, 128, 8, 5, 64, 400000), 47069184), ((80, 64, 32, 32, 32, 2, 1, 64, 5000), 366592),
          ((160, 128, 64, 64, 128, 3, 2, 7, 123457), 9205760), ((33, 17, 10, 11, 12, 1, 4, 1, 0), 21248)]


@pytest.mark.parametrize("shape,before", _SIZES)
def test_workspace_unchanged_without_the_flag(shape, before):
    for flags in (0, N.SPSG_FLAG_RECORD_HITS | N.SPSG_FLAG_VIEW_NORMALS, N.SPSG_FLAG_DETERMINISTIC_GRADS):
        assert N.lib.spsg_workspace_bytes(ctypes.byref(_params(*shape, flags))) == before
    w, h, b, f = shape[0], shape[1], shape[5], shape[6]
    partials = -(-b * f * w * h // 4096) * 64
    det = N.lib.spsg_workspace_bytes(ctypes.byref(_params(*shape, N.SPSG_FLAG_DETERMINISTIC)))
    assert det == before + (partials + 255) // 256 * 256


def test_deterministic_forward_needs_its_workspace():
    """A workspace sized without the flag is refused by a deterministic forward, before anything is enqueued."""
    p = _params(80, 64, 32, 32, 32, 1, 1, 64, 100, N.SPSG_FLAG_DETERMINISTIC)
    small = N.lib.spsg_workspace_bytes(ctypes.byref(_params(80, 64, 32, 32, 32, 1, 1, 64, 100, 0)))
    fake = 1 << 20  # never dereferenced: the size check comes first
    rc = N.lib.spsg_raycast_forward(ctypes.byref(p), *([fake] * 14), fake, small, None)
    assert rc == 3 and b"workspace" in N.lib.spsg_last_error()
    rc = N.lib.spsg_raycast_backward(ctypes.byref(p), *([fake] * 11), fake, small, None)
    assert rc == 3


def test_losses2d_deterministic_validation():
    assert N.lib.spsg_losses2d_deterministic_scratch_bytes(-1) == 0
    assert N.lib.spsg_losses2d_deterministic_scratch_bytes(0) == 4096 + 256
    assert N.lib.spsg_losses2d_deterministic_scratch_bytes(4097) == 4096 + 256 + 256
    fake = 1 << 20
    tg = N.LossTargets(fake, None, None, None, None, 0.02, 1.0, 1.0, 1.0)
    f = N.lib.spsg_losses2d_forward_deterministic
    assert f(None, fake, fake, fake, 10, fake, fake, 1 << 16, None) == 1
    assert f(ctypes.byref(tg), None, None, None, 10, fake, fake, 1 << 16, None) == 1   # depth target without rendering
    assert f(ctypes.byref(tg), None, fake, None, -1, fake, fake, 1 << 16, None) == 1
    assert f(ctypes.byref(tg), None, fake, None, 1 << 20, fake, fake, 4096 + 256, None) == 3
    assert f(ctypes.byref(tg), None, fake, None, 10, fake, fake + 4, 1 << 16, None) == 3  # misaligned scratch


def _sass_functions():
    cuobjdump = shutil.which("cuobjdump") or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")
    if not os.path.isfile(cuobjdump):
        pytest.skip("cuobjdump not found")
    out = subprocess.check_output([cuobjdump, "-sass", N.LIB_PATH], text=True)
    res, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            res[cur] = []
        elif cur is not None:
            res[cur].append(line)
    return res


# what a deterministic call launches besides the fill / index / classification passes: the forward without the fused loss
# epilogue, the canonicalisation and loss kernels, the one-view and view-ordered gathers
_DETERMINISTIC_KERNELS = (r"canon_rows_kernel", r"canon_insert_kernel", r"losses2d_det_kernel", r"raycast_forward_kernelILb0E",
                          r"backward_gather_kernelILb[01]ELb[01]ELi[02]E", r"backward_zero", r"fill_kernel",
                          r"index_(packed_)?kernel", r"cell_class_kernel", r"finalize_loss_kernel")
_FLOAT_ATOMIC = re.compile(r"\b(RED|REDG|REDS|ATOM|ATOMG|ATOMS)\.[\w.]*\b(F16|BF16|F32|F64|F16x2|BF16x2)\b")


def test_deterministic_kernels_have_no_float_atomics():
    funcs = _sass_functions()
    seen = set()
    for name, lines in funcs.items():
        for pat in _DETERMINISTIC_KERNELS:
            if re.search(pat, name):
                seen.add(pat)
                bad = [ln.strip() for ln in lines if _FLOAT_ATOMIC.search(ln)]
                assert not bad, "%s: %s" % (name, bad[:3])
    assert {r"canon_rows_kernel", r"canon_insert_kernel", r"losses2d_det_kernel"} <= seen
    # the pattern does find the default path's float atomics
    assert any(_FLOAT_ATOMIC.search(ln) for name, lines in funcs.items() if "losses2d_forward_kernel" in name for ln in lines)
