"""The one-tile planning kernels, rollout_tc_kernel<1, 4, pair> (the headline) and <1, 4>, must not spill under their
96-register launch bound: their step loop issues every layer as two column halves on double-buffered tensor memory,
which adds per-half hand-off state to kernels already at the register limit. The build compiles with -Xptxas -v
into csrc/*.ptxas.log; this reads that report."""
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LOG = os.path.join(ROOT, 'ethz-safe-learning_b200', 'csrc', 'rollout_tc.o.ptxas.log')
PAIR = '_ZN5simba17rollout_tc_kernelILi1ELi4ELb1EEEvNS_13RolloutParamsE'
ONE_CTA = '_ZN5simba17rollout_tc_kernelILi1ELi4ELb0EEEvNS_13RolloutParamsE'


def _spills(kernel):
    if not os.path.exists(LOG):
        pytest.skip("library not built")
    found = dict((n, (s, l)) for n, s, l in re.findall(
        r"Function properties for (\S+)\n\s*\d+ bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads",
        open(LOG).read()))
    return found.get(kernel)


def test_pair_rollout_kernel_does_not_spill():
    assert _spills(PAIR) == ('0', '0')


def test_one_cta_rollout_kernel_does_not_spill():
    assert _spills(ONE_CTA) == ('0', '0')
