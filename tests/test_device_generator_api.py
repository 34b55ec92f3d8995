"""CPU: DeviceGenerator is public and keeps its state on a CUDA device only."""
import pytest

import nfb200 as N


def test_device_generator_is_exported():
    assert "DeviceGenerator" in N.__all__
    assert N.DeviceGenerator is N.flows.DeviceGenerator


@pytest.mark.parametrize("device", ["cpu", "meta"])
def test_device_generator_refuses_a_non_cuda_device(device):
    with pytest.raises(RuntimeError, match="CUDA memory"):
        N.DeviceGenerator(device)
