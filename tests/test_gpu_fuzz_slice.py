"""A seeded slice of the randomised hunts (tests/fuzz_*.py) under pytest, so that the round-end GPU run sees them: random
grids from 3^3 to 230^3, increments, depth ranges, thresholds, cameras, voxel soups -- and large images that reach the
large-launch instantiation of the forward kernel."""
import pytest

pytestmark = pytest.mark.gpu


def _need_ref():
    from oracle import ref_driver
    if not ref_driver.available(pinned=True):
        pytest.skip("oracle/_ref not built (run __graft_entry__.build() where /root/reference exists)")


def test_fuzz_forward_bit_exact_slice(cuda_device):
    _need_ref()
    from tests import fuzz_parity
    assert fuzz_parity.run(cases=200, seed0=20261, dev=cuda_device, pinned=True) == 0


def test_fuzz_forward_bit_exact_large_images(cuda_device):
    _need_ref()
    from tests import fuzz_parity
    assert fuzz_parity.run(cases=24, seed0=977, dev=cuda_device, large=True, pinned=True) == 0


def test_fuzz_backward_slice(cuda_device):
    _need_ref()
    from tests import fuzz_backward
    assert fuzz_backward.run(cases=80, seed0=31, dev=cuda_device, pinned=True) == 0


def test_fuzz_fused_losses_slice(cuda_device):
    from tests import fuzz_fused
    assert fuzz_fused.run(cases=60, seed0=47, dev=cuda_device) == 0


def test_fuzz_alternative_routes_slice(cuda_device):
    """host-packed rows and the index + brick written by the compaction pass against the plain int64 route"""
    from tests import fuzz_routes
    assert fuzz_routes.run(cases=120, seed0=5, dev=cuda_device) == 0
