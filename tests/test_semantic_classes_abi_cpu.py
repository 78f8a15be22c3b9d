"""Configurable semantic class count without a GPU: the ctypes mirror of spsg_raycast_params.semantic_channels, the debug
flag, the new entry points and their argument checks (which return before anything is enqueued), the workspace (which
does not depend on C), and the SASS of the C-generic kernels a deterministic call launches."""
import ctypes
import os
import re

import pytest

from spsg_b200 import _native as N

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "spsg_raycast.h")


def _header():
    with open(HEADER) as fh:
        return fh.read()


def _params(flags=0, c=0, n=1000):
    return N.make_params(160, 128, 0.1, 6.0, 1.0, 0.9, 64, 64, 128, 2, 3, 64, n, flags, c)


def test_params_field_replaces_reserved():
    src = _header()
    body = re.search(r"typedef struct spsg_raycast_params \{(.*?)\} spsg_raycast_params;", src, re.S).group(1)
    assert re.search(r"uint32_t\s+semantic_channels;", body) and "reserved" not in body
    assert [f[0] for f in N.Params._fields_][-1] == "semantic_channels"
    assert N.Params.semantic_channels.offset == 60 and ctypes.sizeof(N.Params) == 64


def test_flag_and_limit_match_the_header():
    src = _header()
    m = re.search(r"SPSG_FLAG_GENERIC_SEMANTIC\s*=\s*1u\s*<<\s*(\d+)", src)
    assert m and N.SPSG_FLAG_GENERIC_SEMANTIC == 1 << int(m.group(1)) == 1 << 12
    m = re.search(r"#define SPSG_MAX_SEMANTIC_CHANNELS (\d+)", src)
    assert m and int(m.group(1)) == N.SPSG_MAX_SEMANTIC_CHANNELS == 64


def test_new_symbols_are_declared_and_exported():
    src = _header()
    for name in ("spsg_losses2d_forward_classes", "spsg_losses2d_forward_deterministic_classes",
                 "spsg_losses2d_backward_classes", "spsg_labels_from_render_classes"):
        assert re.search(r"SPSG_API int %s\(" % name, src), name
        assert name in N.EXPORTS
        assert hasattr(N.lib, name)


@pytest.mark.parametrize("flags", [0, N.SPSG_FLAG_DETERMINISTIC, N.SPSG_FLAG_ALL_PIXELS | N.SPSG_FLAG_DETERMINISTIC])
def test_workspace_does_not_depend_on_c(flags):
    base = N.lib.spsg_workspace_bytes(ctypes.byref(_params(flags)))
    assert base > 0
    for c in (1, 2, 13, 14, 15, 41, 64):
        for extra in (0, N.SPSG_FLAG_GENERIC_SEMANTIC):
            assert N.lib.spsg_workspace_bytes(ctypes.byref(_params(flags | extra, c))) == base


@pytest.mark.parametrize("c", [65, 100, 1 << 31])
def test_out_of_range_c_is_rejected(c):
    assert N.lib.spsg_workspace_bytes(ctypes.byref(_params(0, c))) == 0
    assert b"semantic_channels" in N.lib.spsg_last_error()
    fake = 1 << 20  # never dereferenced: the checks return first
    p = _params(0, c)
    assert N.lib.spsg_raycast_forward(ctypes.byref(p), *([fake] * 14), fake, 1 << 30, None) == 1
    assert N.lib.spsg_raycast_backward(ctypes.byref(p), *([fake] * 11), fake, 1 << 30, None) == 1


@pytest.mark.parametrize("c", [0, -1, 65])
def test_standalone_entry_points_check_the_class_count(c):
    fake = 1 << 20
    tg = N.LossTargets(None, None, None, fake, None, 0.02, 1.0, 1.0, 1.0)
    assert N.lib.spsg_losses2d_forward_classes(ctypes.byref(tg), None, None, fake, c, 100, fake, fake, 4096, None) == 1
    assert N.lib.spsg_losses2d_forward_deterministic_classes(ctypes.byref(tg), None, None, fake, c, 100, fake, fake,
                                                             1 << 20, None) == 1
    assert N.lib.spsg_losses2d_backward_classes(ctypes.byref(tg), None, None, fake, c, 100, fake, None, None, None, fake,
                                                None) == 1
    assert N.lib.spsg_labels_from_render_classes(fake, c, 100, fake, None, None) == 1


def test_generic_deterministic_kernels_have_no_float_atomics():
    from tests.test_deterministic_cpu import _FLOAT_ATOMIC, _sass_functions
    funcs = _sass_functions()
    # what a deterministic call launches with kGenericSem: the forward without the fused-loss epilogue, the gathers with one
    # view or view-ordered means (table and segment), the deterministic loss sums, the stand-alone loss backward and the
    # zero kernels
    pats = (r"raycast_forward_kernelILb0ELb[01]ELi\d+ELb[01]ELb1E", r"backward_gather_kernelILb[01]ELb[01]ELi[02]ELb[01]ELb[01]ELb1E",
            r"losses2d_det_kernelILb1E", r"losses2d_backward_kernelILb1E", r"backward_zero_sem_kernel")
    seen = set()
    for name, lines in funcs.items():
        for pat in pats:
            if re.search(pat, name):
                seen.add(pat)
                bad = [ln.strip() for ln in lines if _FLOAT_ATOMIC.search(ln)]
                assert not bad, "%s: %s" % (name, bad[:3])
    assert seen == set(pats)
    # the default-mode variants do have them: the fused forward's loss sums, the several-view gather's means
    assert any(_FLOAT_ATOMIC.search(ln) for name, lines in funcs.items()
               if re.search(r"raycast_forward_kernelILb1ELb0ELi24ELb0ELb1E", name) for ln in lines)
    assert any(_FLOAT_ATOMIC.search(ln) for name, lines in funcs.items()
               if re.search(r"backward_gather_kernelILb0ELb0ELi1ELb0ELb0ELb1E", name) for ln in lines)
