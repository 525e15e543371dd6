"""The bf16 forward entry points are declared, exported and bound, and without a GPU they fail with a device error
instead of running anything on the CPU."""
import ctypes as C

import pytest

from tests.test_abi import declared_functions

NAMES = ('simba_ensemble_forward_tc', 'simba_ensemble_forward_tc_kernel')


def test_forward_tc_symbols_are_declared_exported_and_bound():
    from simba_b200 import _lib
    lib = _lib.load()
    for name in NAMES:
        assert name in declared_functions()
        assert name in _lib.exported_names()
        assert hasattr(lib, name)


def test_forward_tc_without_gpu_returns_a_device_error():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from simba_b200 import _lib
    lib = _lib.load()
    k, items = C.c_int32(-1), C.c_int32(-1)
    assert lib.simba_ensemble_forward_tc_kernel(None, 3000, C.byref(k), C.byref(items)) in (-3, -5)
    assert (k.value, items.value) == (-1, -1)
    assert lib.simba_ensemble_forward_tc(None, None, None, 3000, None, None, None, None) in (-3, -5)
    assert lib.simba_last_error()


def test_precision_is_keyword_only_and_checked_before_any_device_work():
    from simba_b200.models import MlpEnsemble
    ens = MlpEnsemble(4, 3, 2, mlp_params=dict(n_layers=1, units=8))
    x = [[0.0] * 4] * 2
    with pytest.raises(TypeError):
        ens.forward(x, 'bf16')
    for bad in ('fp16', 'BF16', None):
        with pytest.raises(ValueError):
            ens.forward(x, precision=bad)
        with pytest.raises(ValueError):
            ens(x, None, precision=bad)
