"""The weight-streaming tcgen05 kernel (both state widths) must not spill: its 18-warp CTA caps it at 96 registers,
and the 128-column variant stays under that only because it re-derives its scorer predicates every step. The
build compiles with -Xptxas -v into csrc/*.ptxas.log; this reads that report."""
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LOG = os.path.join(ROOT, 'ethz-safe-learning_b200', 'csrc', 'rollout_tc_wide.o.ptxas.log')


def test_streaming_rollout_kernels_do_not_spill():
    if not os.path.exists(LOG):
        pytest.skip("library not built")
    text = open(LOG).read()
    found = re.findall(r"Function properties for (\S*rollout_tc_wide_kernel\S*)\n\s*\d+ bytes stack frame, "
                       r"(\d+) bytes spill stores, (\d+) bytes spill loads", text)
    assert sorted(n for n, _, _ in found) == ['_ZN5simba22rollout_tc_wide_kernelILi128EEEvNS_13RolloutParamsE',
                                              '_ZN5simba22rollout_tc_wide_kernelILi64EEEvNS_13RolloutParamsE']
    for name, stores, loads in found:
        assert (stores, loads) == ('0', '0'), name
