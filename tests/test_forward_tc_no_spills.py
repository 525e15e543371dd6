"""The forward forms of the tcgen05 rollout kernels (simba_ensemble_forward_tc) must not spill. The build compiles
with -Xptxas -v into csrc/*.ptxas.log; this reads that report for every instantiation."""
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, 'ethz-safe-learning_b200', 'csrc')
EXPECTED = {
    'rollout_tc.o.ptxas.log': ['_ZN5simba17forward_tc_kernelILi1ELi4EEEvNS_13RolloutParamsE',
                               '_ZN5simba17forward_tc_kernelILi2ELi2EEEvNS_13RolloutParamsE'],
    'rollout_tc_wide.o.ptxas.log': ['_ZN5simba22forward_tc_wide_kernelILi128EEEvNS_13RolloutParamsE',
                                    '_ZN5simba22forward_tc_wide_kernelILi64EEEvNS_13RolloutParamsE'],
}


@pytest.mark.parametrize("log", list(EXPECTED))
def test_forward_kernels_do_not_spill(log):
    path = os.path.join(CSRC, log)
    if not os.path.exists(path):
        pytest.skip("library not built")
    found = re.findall(r"Function properties for (\S*forward_tc\S*)\n\s*\d+ bytes stack frame, "
                       r"(\d+) bytes spill stores, (\d+) bytes spill loads", open(path).read())
    assert sorted(n for n, _, _ in found) == EXPECTED[log]
    for name, stores, loads in found:
        assert (stores, loads) == ('0', '0'), name
