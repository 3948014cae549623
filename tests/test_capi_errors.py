"""Failures of the C ABI reach Python with the message vgsim_last_error() holds.  Without a CUDA device every device
allocation fails, which makes the error path of the sampler taps reachable on a CPU-only machine."""
import numpy as np
import pytest

from vgsim_b200 import _capi


def _has_gpu():
    import torch
    return torch.cuda.is_available()


@pytest.mark.skipif(_has_gpu(), reason="needs a machine without a CUDA device")
@pytest.mark.parametrize("call", [
    lambda: _capi.test_poisson([1.0]),
    lambda: _capi.test_hypergeometric([5], [5], [3], np.arange(16, dtype=np.uint64)),
    lambda: _capi.test_choose([1.0, 2.0], [0.5]),
], ids=["poisson", "hypergeometric", "choose"])
def test_tap_failure_carries_the_cuda_error(call):
    with pytest.raises(_capi.VgsimError) as err:
        call()
    msg = str(err.value)
    assert msg == _capi.lib.vgsim_last_error().decode()
    assert msg.startswith("cudaMalloc: ") and len(msg) > len("cudaMalloc: ")
