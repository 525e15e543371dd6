"""The swish kernels' ptxas reports (-Xptxas -v, csrc/*.ptxas.log). Every swish instantiation is listed here with the
spill bytes it compiles to; most spill nothing.

The exceptions sit at the 96-register bound of the 16-warp tcgen05 CTA (kBoundThreads), where the ReLU kernels
already are: the swish drain keeps each 32-column accumulator load live through its tanh.approx operations.
  * rollout_swish_tc_kernel<2, 2>: 28 / 48 bytes, exactly what the ReLU rollout_tc_kernel<2, 2> spills.
  * rollout_swish_tc_kernel<1, 4, false>, unfold_swish_tc_kernel<2, 2>, forward_swish_tc_kernel<2, 2>: 16-28
    bytes of stores. Splitting the drain's stores and packing the arithmetic as f32x2 were tried and spill as
    much or more.
  * train_swish_chain_kernel<4>: 8 bytes, the accurate expf of swish and swish' next to the 4-row tile.
The limits below are the measured values: a change that spills more fails here."""
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, 'ethz-safe-learning_b200', 'csrc')

# log -> {kernel name pattern: (max spill store bytes, max spill load bytes)}
EXPECTED = {
    'rollout_f32.o.ptxas.log': {r'rollout_swish_f32_kernel': (0, 0)},
    'rollout_tc.o.ptxas.log': {
        r'rollout_swish_tc_kernelILi1ELi4ELb1E': (0, 0),
        r'rollout_swish_tc_kernelILi1ELi4ELb0E': (20, 24),
        r'rollout_swish_tc_kernelILi2ELi2ELb0E': (28, 48),
        r'unfold_swish_tc_kernelILi1ELi4E': (0, 0),
        r'unfold_swish_tc_kernelILi2ELi2E': (16, 32),
        r'forward_swish_tc_kernelILi1ELi4E': (0, 0),
        r'forward_swish_tc_kernelILi2ELi2E': (28, 44),
    },
    'rollout_tc_wide.o.ptxas.log': {
        r'%s_swish_tc_wide_kernelILi%dE' % (form, sw): (0, 0)
        for form in ('rollout', 'unfold', 'forward') for sw in (64, 128)},
    'trainer_f32.o.ptxas.log': {r'train_swish_chain_kernelILi4E': (8, 4), r'train_swish_chain_kernelILi8E': (0, 0),
                                r'train_swish_chain_kernelILi16E': (0, 0)},
    'trainer_tc.o.ptxas.log': {r'train_swish_tc_chain_kernel': (0, 0)},
}


@pytest.mark.parametrize("log", list(EXPECTED))
def test_swish_kernels_spill_no_more_than_recorded(log):
    path = os.path.join(CSRC, log)
    if not os.path.exists(path):
        pytest.skip("library not built")
    found = re.findall(r"Function properties for (\S*swish\S*)\n\s*\d+ bytes stack frame, "
                       r"(\d+) bytes spill stores, (\d+) bytes spill loads", open(path).read())
    assert len(found) == len(EXPECTED[log])
    for pattern, (max_st, max_ld) in EXPECTED[log].items():
        hits = [(int(s), int(l)) for n, s, l in found if re.search(pattern, n)]
        assert len(hits) == 1, pattern
        assert hits[0][0] <= max_st and hits[0][1] <= max_ld, (pattern, hits[0])
