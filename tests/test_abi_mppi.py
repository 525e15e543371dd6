"""The MPPI update rule's C surface: the enum matches ctypes, the setter and the per-kernel entry point are declared,
exported and bound, and they reject a null planner before touching a device."""
import pytest

from tests.test_abi import _print_from_c, declared_functions

NAMES = ('simba_planner_set_update_rule', 'simba_mppi_update')


def test_update_rule_constants_match_ctypes():
    from simba_b200 import _lib
    assert _print_from_c('%d %d', '(int)SIMBA_UPDATE_CEM', '(int)SIMBA_UPDATE_MPPI') == [_lib.UPDATE_CEM,
                                                                                       _lib.UPDATE_MPPI]


def test_mppi_symbols_are_declared_exported_and_bound():
    from simba_b200 import _lib
    lib = _lib.load()
    for name in NAMES:
        assert name in declared_functions()
        assert name in _lib.exported_names()
        assert hasattr(lib, name)


def test_null_planner_is_a_config_error():
    from simba_b200 import _lib
    lib = _lib.load()
    assert lib.simba_planner_set_update_rule(None, _lib.UPDATE_MPPI, 1.0) == -1
    assert lib.simba_mppi_update(None, None, None, None, None, None, None, None) == -1
    assert lib.simba_last_error()


def test_mppi_policies_take_no_elite_options():
    import inspect
    from simba_b200.policies import MppiMpc, SafeMppiMpc
    for cls in (MppiMpc, SafeMppiMpc):
        params = inspect.signature(cls.__init__).parameters
        assert 'temperature' in params and 'n_elite' not in params and 'stddev_threshold' not in params
    with pytest.raises(ValueError):
        SafeMppiMpc(None, None, 5, 2, 0.0, 10, 2, 0.01, 1.0, 0.1, selection='feasible_first')
