"""The bf16 unfold entry points are declared, exported and bound, and without a GPU they fail with a device
error instead of running anything on the CPU."""
import ctypes as C

import pytest

from tests.test_abi import declared_functions

NAMES = ('simba_unfold_tc', 'simba_unfold_tc_kernel')


def test_unfold_tc_symbols_are_declared_exported_and_bound():
    from simba_b200 import _lib
    lib = _lib.load()
    for name in NAMES:
        assert name in declared_functions()
        assert name in _lib.exported_names()
        assert hasattr(lib, name)


def test_unfold_tc_without_gpu_returns_a_device_error():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from simba_b200 import _lib
    lib = _lib.load()
    k, items = C.c_int32(-1), C.c_int32(-1)
    assert lib.simba_unfold_tc_kernel(None, 3000, 15, C.byref(k), C.byref(items)) in (-3, -5)
    assert (k.value, items.value) == (-1, -1)
    assert lib.simba_unfold_tc(None, None, None, None, 0, 3000, 15, 1, None, None) in (-3, -5)
    assert lib.simba_last_error()
