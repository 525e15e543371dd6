"""The MPPI kernels (mppi_update_kernel<staged>, mppi_refit_kernel, mppi_finalize_kernel) must not spill. The build compiles with
-Xptxas -v into csrc/*.ptxas.log; this reads cem_kernels.o's report."""
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LOG = os.path.join(ROOT, 'ethz-safe-learning_b200', 'csrc', 'cem_kernels.o.ptxas.log')
KERNELS = ('_ZN5simba18mppi_update_kernelILb0EEEvNS_16MppiUpdateParamsE',
           '_ZN5simba18mppi_update_kernelILb1EEEvNS_16MppiUpdateParamsE',
           '_ZN5simba17mppi_refit_kernelENS_10MppiParamsEii',
           '_ZN5simba20mppi_finalize_kernelENS_14FinalizeParamsEi')


def test_mppi_kernels_do_not_spill():
    if not os.path.exists(LOG):
        pytest.skip("library not built")
    found = dict((n, (int(s), int(l))) for n, s, l in re.findall(
        r"Function properties for (\S*mppi_\S*)\n\s*\d+ bytes stack frame, (\d+) bytes spill stores, "
        r"(\d+) bytes spill loads", open(LOG).read()))
    assert sorted(found) == sorted(KERNELS)
    for name in KERNELS:
        assert found[name] == (0, 0), name
