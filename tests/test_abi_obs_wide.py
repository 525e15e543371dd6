"""The wide-observation rollout kernel's constant: include/simba_b200.h and simba_b200/_lib.py agree."""
from tests.test_abi import _print_from_c


def test_wide_observation_kernel_constant_matches_ctypes():
    from simba_b200 import _lib
    assert _print_from_c('%d', '(int)SIMBA_ROLLOUT_TC_WIDE_OBS') == [_lib.ROLLOUT_TC_WIDE_OBS]
    assert _lib.ROLLOUT_TC_WIDE_OBS == 5
