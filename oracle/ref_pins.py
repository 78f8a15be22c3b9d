"""Recorded outputs of the reference extensions, for checkouts where they are not built (test infrastructure only).

``tests/golden/ref_pins.json`` maps every native call the parity tests make on the reference's entry points
(``raycast_rgbd_cuda`` and ``depth_utils_cuda``) to what the call wrote.  Deterministic outputs (renderings,
registration counts, pixel tables, index, depth maps) are kept as a digest, so they are checked bit for bit.  Voxel
gradients, which the reference accumulates with float atomics in arbitrary order, are kept as seeded random-weight dot
products (a gradient routed to the wrong voxel or a dropped pixel contribution moves them) and a seeded sample of
their non-zero entries, checked at the tests' bar of 1e-3 of the largest magnitude.  A call is identified by a digest
of its name, its input tensors and its scalars; inputs the tests draw on the GPU make the keys depend on torch's
random number generators, so a torch release that changes them invalidates the table.

Where ``oracle/_ref`` is not built, ``stand_in`` takes the reference module's place for tests that ask for it: it runs
each call on this package's drop-in module of the same name and signature and asserts that the outputs are the
recorded ones.  A call that was never recorded fails.

    SPSG_REF_PINS_RECORD=<file> python -m pytest tests -m gpu      (with oracle/_ref built)

records the table from the compiled reference extensions and writes <file> at exit.

Provenance of the committed table: the reference's sources are not part of this repository, and the table was
recorded through the drop-in modules at commit c678dcf.  Its CUDA sources, package and tests are identical to those
of commit a7e897c, whose GPU suite, these parity tests included, passed against the compiled reference extensions
(GPUTEST_r02.json in commit 1201976: 101 passed).  Record it again from the extensions wherever they can be built.
"""
import atexit
import hashlib
import json
import os

import numpy as np
import torch

PINS = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "ref_pins.json")
RECORD = os.environ.get("SPSG_REF_PINS_RECORD")
GRAD_DOTS = 4       # random-weight dot products per gradient tensor
GRAD_SAMPLES = 4    # non-zero entries sampled per gradient tensor
GRAD_RTOL = 1e-3    # of the tensor's largest magnitude, per entry (the parity tests' bar)

# kind -> name -> (input argument positions, output argument positions); the reference's signatures
SIGNATURES = {
    "raycast": {
        "construct_dense_sparse_mapping": ((0,), (1,)),
        "forward": ((1, 2, 3, 4, 5, 6, 13, 14), (0, 7, 8, 9, 10, 11, 12)),
        "backward": ((0, 1, 2, 3, 4, 6, 7), (8, 9, 10, 11)),
        "raycast_occ": ((0, 2, 3, 4), (1,)),
    },
    "depth": {
        "bilateral_filter_floatmap": ((1, 2, 3), (0,)),
        "median_fill_depthmap": ((1,), (0,)),
        "convert_depth_to_cameraspace": ((1, 2, 3, 4), (0,)),
        "compute_normals": ((1,), (0,)),
    },
}

_table = None
_recorded = {}


def recorded():
    return os.path.isfile(PINS)


def _load():
    global _table
    if _table is None:
        with open(PINS) as f:
            _table = json.load(f)["calls"]
    return _table


def _update(h, a):
    if isinstance(a, torch.Tensor):
        t = a.detach().contiguous().cpu()
        h.update(("%s%s" % (t.dtype, tuple(t.shape))).encode())
        h.update(t.view(torch.uint8).numpy().tobytes() if t.numel() else b"")
    else:
        h.update(repr(a).encode())


def _mapping_canonical(mapping, num):
    """mapping3dto2d with each row's registered pixels sorted and the unused tail blanked; rows whose voxel overflowed
    max_pixels_per_voxel keep an arbitrary subset in the reference and are blanked whole."""
    max_pix = mapping.shape[1]
    num = num.view(-1, 1).long()
    used = torch.arange(max_pix, device=mapping.device).view(1, -1) < num
    rows = torch.where(used, mapping, torch.full_like(mapping, torch.iinfo(mapping.dtype).max)).sort(dim=1).values
    return torch.where(num > max_pix, torch.full_like(rows, -1), rows)


def _weights(size):
    return np.random.default_rng(size).uniform(-1.0, 1.0, (GRAD_DOTS, size))


def _grad_summary(t, n):
    """[largest magnitude, non-zero count, GRAD_DOTS dot products, GRAD_SAMPLES x (flat index, value) of non-zeros]"""
    t = t[:n].detach().double().cpu().numpy().ravel()
    nz = np.flatnonzero(t)
    pick = np.random.default_rng(t.size + 1).choice(nz, size=min(GRAD_SAMPLES, nz.size), replace=False)
    r = lambda x: float("%.9g" % x)
    out = [r(np.abs(t).max()) if t.size else 0.0, int(nz.size)] + [r(d) for d in _weights(t.size) @ t]
    for i in pick:
        out += [int(i), r(t[i])]
    return out


def _grad_check(t, n, want):
    """The entries within GRAD_RTOL of the recorded largest magnitude; each dot product within what such entry errors
    could add up to at random (GRAD_RTOL x largest magnitude x sqrt(non-zero count))."""
    t = t[:n].detach().double().cpu().numpy().ravel()
    vmax, nnz, dots, pairs = want[0], want[1], want[2:2 + GRAD_DOTS], want[2 + GRAD_DOTS:]
    tol = GRAD_RTOL * vmax
    if abs(float(np.abs(t).max()) - vmax) > tol if t.size else vmax != 0:
        return False
    if any(abs(t[int(i)] - v) > tol for i, v in zip(pairs[0::2], pairs[1::2])):
        return False
    got = _weights(t.size) @ t
    return all(abs(g - d) <= tol * max(1.0, np.sqrt(nnz)) for g, d in zip(got, dots))


class PinnedModule:
    """A native module of the reference's signature whose calls are checked against (``record``: recorded into) the
    table."""

    def __init__(self, impl, kind, record=False):
        self._impl, self._sigs, self._record = impl, SIGNATURES[kind], record

    def __getattr__(self, name):
        if name not in self._sigs:
            raise AttributeError(name)
        inputs, outputs = self._sigs[name]

        def call(*args):
            key = hashlib.sha256(name.encode())
            for i in inputs:
                _update(key, args[i])
            key = key.hexdigest()[:24]
            result = getattr(self._impl, name)(*args)
            outs = [args[i] for i in outputs]
            if name == "backward":
                n = int(args[7][4])
                # a voxel seen by more pixels than its table holds gets gradients from an arbitrary subset of them in
                # the reference: not pinned (the tests skip such cases too)
                overflow = n and int(args[6][:n].max()) > args[5].shape[1]
                if self._record:
                    _recorded[key] = "overflow" if overflow else [_grad_summary(t, n) for t in outs]
                    return result
                want = _load().get(key)
                assert want is not None, "reference backward: no recorded output for these inputs (%s)" % PINS
                assert bool(overflow) == (want == "overflow"), "reference backward: pixel-table overflow differs"
                assert overflow or all(_grad_check(t, n, w) for t, w in zip(outs, want)), \
                    "reference backward: gradients differ from the recorded reference gradients"
                return result
            if name == "forward":  # one view per call: rows [0, N) of the registration tables are this call's
                n = args[1].shape[0]
                outs[5], outs[6] = _mapping_canonical(outs[5][:n], outs[6][:n]), outs[6][:n]
            h = hashlib.sha256()
            for t in outs:
                _update(h, t)
            got = h.hexdigest()[:24]
            if self._record:
                _recorded[key] = got
                return result
            want = _load().get(key)
            assert want is not None, "reference %s: no recorded output for these inputs (%s)" % (name, PINS)
            assert got == want, "reference %s: outputs differ from the recorded reference outputs" % name
            return result
        return call


def stand_in(kind):
    """The reference module of ``kind`` ("raycast" or "depth") where it is not built: the drop-in module, checked."""
    if kind == "raycast":
        from spsg_b200.dropin import raycast_rgbd_cuda as impl
    else:
        from spsg_b200.dropin import depth_utils_cuda as impl
    return PinnedModule(impl, kind)


def write(path):
    if _recorded:
        with open(path, "w") as f:
            json.dump({"calls": dict(sorted(_recorded.items()))}, f, separators=(",", ":"))
            f.write("\n")


if RECORD:
    atexit.register(write, RECORD)
