"""The bf16 tcgen05 trainer kernels must not spill. The build compiles with -Xptxas -v into
csrc/*.ptxas.log; this reads trainer_tc.o's report."""
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LOG = os.path.join(ROOT, 'ethz-safe-learning_b200', 'csrc', 'trainer_tc.o.ptxas.log')


def test_bf16_trainer_kernels_do_not_spill():
    if not os.path.exists(LOG):
        pytest.skip("library not built")
    text = open(LOG).read()
    found = re.findall(r"Function properties for (\S*train_tc_\w+_kernel\S*)\n\s*\d+ bytes stack frame, "
                       r"(\d+) bytes spill stores, (\d+) bytes spill loads", text)
    assert sorted(re.search(r'train_tc_\w+_kernel', n).group(0) for n, _, _ in found) == \
        ['train_tc_chain_kernel', 'train_tc_update_kernel']
    for name, stores, loads in found:
        assert (stores, loads) == ('0', '0'), name
