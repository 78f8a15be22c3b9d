#!/usr/bin/env python
"""Generate tests/golden/frame_io_ref.npz with the reference's OWN `data_util.load_frames` (needs baseline/_ref, CPU).

    python tests/golden/make_golden_frame_io.py

For every case of tests/test_frame_io_cpu.py the test's synthetic frame files are written to a temporary directory and
the reference's outputs on them stored: depth and colour (as SHA-256 digests), poses, intrinsics and frame ids of the
two-frame call, depth (digest) and intrinsics of the 'self' / depth-only call.  tests/test_frame_io_cpu.py compares frame_io with them where baseline/_ref
is not installed.

Provenance of the committed file: the reference's sources are not part of this repository; it was written from
frame_io.load_frames at commit c678dcf, which DESIGN.md section 6a records as bit-identical to the reference's function
on exactly these files (the comparison this test makes when baseline/_ref is installed).  Regenerate it here wherever
baseline/_ref can be installed."""
import os
import pathlib
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from tests import test_frame_io_cpu as T  # noqa: E402


def main(du):
    out = {}
    for src_wh, dst_wh in T.CASES:
        with tempfile.TemporaryDirectory() as d:
            _, _, want, want_self = T.reference_outputs(du, pathlib.Path(d), src_wh, dst_wh)
        k = T._golden_key(src_wh, dst_wh)
        out[k + "_depth"], out[k + "_color"] = T.digest(want[0]), T.digest(want[1])
        out[k + "_pose"], out[k + "_intr"] = want[2].numpy(), want[3].numpy()
        out[k + "_frameids"] = np.array([list(f) for f in want[4]], dtype=np.int64)
        out[k + "_self_depth"], out[k + "_self_intr"] = T.digest(want_self[0]), want_self[3].numpy()
    np.savez_compressed(T.GOLDEN, **out)
    print("wrote", T.GOLDEN, os.path.getsize(T.GOLDEN), "bytes")


if __name__ == "__main__":
    du = T._reference_data_util()
    if du is None:
        raise SystemExit("baseline/_ref is not installed: the reference's data_util is needed")
    main(du)
