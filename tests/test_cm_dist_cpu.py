"""CPU: DistributedClusterMemory's C entry (reid_cm_forward_push) validates its arguments before any CUDA call, the ABI
version names it, and the module has ClusterMemory's surface plus `group`."""
import ctypes
import inspect

import pytest
import torch


def test_abi_version_is_5():
    from reid_gan_b200 import _lib
    assert _lib.lib().reid_abi_version() == 5


def test_forward_push_argument_validation():
    from reid_gan_b200 import _lib
    L = _lib.lib()
    buf = (ctypes.c_int64 * 16)()
    a = ctypes.addressof(buf)

    def push(B=8, D=64, me=0, world=2, cap=8, base=a, inputs=a, B_split=16):
        return L.reid_cm_forward_push(inputs, a, a, B, 5, D, 0.05, B_split, a, a, a, a, a, me, world, cap, base, None)

    for kw, what in [(dict(inputs=None), "NULL"), (dict(base=None), "NULL"), (dict(me=2), "rank"),
                     (dict(me=-1), "rank"), (dict(B=9), "cap"), (dict(B=9, cap=9, B_split=8), "B_split"),
                     (dict(D=4097), "D=4097"), (dict(B=0), "shape")]:
        rc = push(**kw)
        assert rc == _lib.REID_ERR_INVALID_ARG, kw
        assert what in _lib.last_error(), (kw, _lib.last_error())


def test_constructor_is_cluster_memory_plus_group():
    import reid_gan_b200 as rg
    base = list(inspect.signature(rg.ClusterMemory.__init__).parameters)
    sig = inspect.signature(rg.DistributedClusterMemory.__init__)
    assert list(sig.parameters) == base + ["group"]
    assert sig.parameters["group"].default is None
    assert list(inspect.signature(rg.DistributedClusterMemory.forward).parameters)[1:] == [
        "inputs", "targets", "gan_inputs", "conf_weight"]
    assert issubclass(rg.DistributedClusterMemory, rg.ClusterMemory)
    m = rg.DistributedClusterMemory(32, 5)
    assert m.features.shape == (5, 32) and m.gan_features.shape == (5, 32) and m.temp == 0.05 and m.momentum == 0.2
    assert m.group is None


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_no_cpu_fallback():
    import reid_gan_b200 as rg
    x, _ = rg.synth(16, 32, 4)
    with pytest.raises(RuntimeError):
        rg.DistributedClusterMemory(32, 4)(x[:8], torch.zeros(8, dtype=torch.long))
