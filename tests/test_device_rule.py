"""The device rule of the Python entry points (_lib.input_device / on_input_device) on the host: which devices a call's
arguments name, the error for CUDA inputs on different devices, and that calls without CUDA inputs leave the current
device alone.  The same rule on real devices is checked in test_gpu_multidevice.py."""
import pytest
import torch


class _OnDevice(object):
    """stands in for an input that is not a tensor but lives on a device (network.SplitCostVolume)"""

    def __init__(self, dev):
        self.device = torch.device(dev)


def _lib():
    import atvsnet_b200 as A
    return A._lib


def test_inputs_on_different_devices_raise():
    L = _lib()
    with pytest.raises(ValueError, match=r'different devices \(cuda:0, cuda:1\)'):
        L.input_device([_OnDevice('cuda:0'), {'x': (_OnDevice('cuda:1'),)}])


def test_decorated_call_without_cuda_inputs_runs_unchanged():
    L = _lib()
    calls = []

    @L.on_input_device
    def op(x, scale=1.0, name='op'):
        """doc"""
        calls.append((x, scale, name))
        return x * scale

    assert op.__name__ == 'op' and op.__doc__ == 'doc'
    assert torch.equal(op(torch.ones(2), scale=2.0), torch.full((2,), 2.0))
    assert len(calls) == 1


def test_decorated_call_with_mixed_devices_never_runs():
    L = _lib()
    calls = []

    @L.on_input_device
    def op(a, b):
        calls.append(1)

    with pytest.raises(ValueError, match='op: CUDA inputs on different devices'):
        op(_OnDevice('cuda:1'), [_OnDevice('cuda:2')])
    assert calls == []
