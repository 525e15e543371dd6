"""CPU-side checks of the drop-in boundary: the header is plain C, the shared object loads and
exports every symbol include/simba_b200.h declares, ctypes structs match the C layout, and — with
no GPU — compute entry points fail loudly instead of falling back to a CPU path."""
import ctypes as C
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, 'include', 'simba_b200.h')


def declared_functions():
    src = open(HEADER).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    return sorted(set(re.findall(r'\b(simba_[a-z0-9_]+)\s*\(', src)))


def test_header_declares_the_expected_surface():
    names = declared_functions()
    for must in ('simba_plan', 'simba_plan_host', 'simba_sample_actions', 'simba_rollout_score',
                 'simba_score_reduce', 'simba_allgather_scores', 'simba_select_elites', 'simba_refit',
                 'simba_unfold', 'simba_ensemble_forward', 'simba_model_set_layer'):
        assert must in names


def test_library_loads_and_exports_every_declared_symbol():
    from simba_b200 import _lib
    lib = _lib.load()
    for name in declared_functions():
        assert hasattr(lib, name), name
    assert sorted(_lib.exported_names()) == declared_functions()
    assert b'sm_100a' in lib.simba_version()


def _print_from_c(fmt, *args):
    """Compile and run `printf(fmt, args...)` as a C99 program that includes the header -> the integers printed."""
    prog = '#include <stdio.h>\n#include "simba_b200.h"\nint main(void) { printf("%s\\n", %s); return 0; }\n' % (
        fmt, ', '.join(args))
    with tempfile.TemporaryDirectory() as d:
        src = os.path.join(d, 't.c')
        open(src, 'w').write(prog)
        exe = os.path.join(d, 't')
        subprocess.check_call(['gcc', '-std=c99', '-Wall', '-Werror', '-I', os.path.join(ROOT, 'include'),
                               src, '-o', exe])
        return [int(v) for v in subprocess.check_output([exe]).split()]


def test_header_is_plain_c_and_struct_sizes_match_ctypes():
    from simba_b200 import _lib
    sizes = _print_from_c('%zu %zu %zu', 'sizeof(simba_model_config_t)', 'sizeof(simba_scorer_t)',
                          'sizeof(simba_planner_config_t)')
    assert sizes == [C.sizeof(_lib.ModelConfig), C.sizeof(_lib.Scorer), C.sizeof(_lib.PlannerConfig)]


def test_rollout_kernel_constants_match_ctypes():
    from simba_b200 import _lib
    names = ('FP32', 'TC_ONE_CTA', 'TC_PAIR', 'TC_TWO_TILE', 'TC_WIDE')
    values = _print_from_c(' '.join(['%d'] * len(names)), *['(int)SIMBA_ROLLOUT_' + n for n in names])
    assert values == [getattr(_lib, 'ROLLOUT_' + n) for n in names]


def test_no_cpu_fallback_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from simba_b200 import SimbaError, _lib
    from tests import helpers
    lib = _lib.load()
    assert lib.simba_device_check() != 0
    cfg = _lib.ModelConfig(60, 2, 5, 4, 128)
    h = C.c_void_p()
    assert lib.simba_model_create(C.byref(cfg), C.byref(h)) in (-3, -5)
    assert lib.simba_last_error()
    c = helpers.workload('tiny')
    pol = helpers.cuda_policy(c, 'penalty')
    with pytest.raises(SimbaError):
        pol.generate_action(c['state'])


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, 'ethz-safe-learning_b200')
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.h')):
                text = open(os.path.join(dirpath, f)).read()
                assert 'import oracle' not in text and 'from oracle' not in text, f
