"""The one-tile rollout kernels (the CTA pair and the one-CTA kernel) issue every layer as two 64-column halves on
double-buffered tensor memory, and the pair multiplies only its own head columns. Their rows must stay bit-identical
to the same rows run batched through the two-tile kernel, which issues whole N = 128 layers: the accumulation order
per output element is the same (K-steps 0..7, then the bias).

Depths 1, 2 and 3 cover both parities of the GEMM count per step (L + 1), so the buffer a step starts on alternates
or not; narrow hidden layers (U < 128) run zero-padded. At depth 5 neither the two-tile nor the pair kernel fits in
shared memory: there the batched launch is the persistent one-CTA kernel walking several work items, against the
same kernel on one state at a time. Both propagation modes, external draws and the kernels' own Philox draws (whose
counters hold the state index, so only the first state's rows can be compared alone).
"""
import numpy as np
import pytest

from tests import helpers
from tests.test_gpu_dispatch_variants import SEED64, _library_choice, _set_switches, _sms, _tc_variant, _tiles
from tests.test_gpu_kernels import dev, P

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

CASES = {                     # name: workload overrides
    'L1': dict(L=1),
    'L2-U96': dict(L=2, U=96),
    'L3': dict(L=3),
    'L3-U40': dict(L=3, U=40),
    'L5': dict(L=5),
}


def _rollout(c, acts, eps, sampling, seed=0, it=0):
    """One simba_rollout_score call of a fresh bf16 planner -> (return, cost mask, cost sum), each [S, P*N]."""
    from simba_b200 import _lib
    lib = _lib.load()
    pol = helpers.cuda_policy(c, 'penalty', precision='bf16', sampling_propagation=sampling)
    pl = pol._ensure_planner()
    S, B = c['S'], c['P'] * c['N']
    ret = torch.full((S * B,), np.nan, dtype=torch.float32, device='cuda')
    mask = torch.full((S * B,), -1, dtype=torch.int64, device='cuda')
    csum = torch.full((S * B,), np.nan, dtype=torch.float32, device='cuda')
    d_state = dev(np.asarray(c['state'], np.float32).reshape(S, c['O']))
    d_eps = dev(eps) if eps is not None else None
    _lib.check(lib.simba_rollout_score(pl, P(d_state), P(dev(acts)), P(d_eps), seed, it, None, P(ret), P(mask),
                                       P(csum), None))
    torch.cuda.synchronize()
    return tuple(x.cpu().numpy().reshape(S, B) for x in (ret, mask, csum))


@pytest.mark.parametrize("sampling", [True, False], ids=['sampling', 'mean'])
@pytest.mark.parametrize("case", list(CASES))
def test_one_tile_rows_equal_batched_rows(case, sampling, monkeypatch):
    over = CASES[case]
    c1 = helpers.workload('c1', **over)
    sms = _sms()
    S = next(S for S in range(1, 64) if len(_tiles(dict(c1, S=S))) > sms)   # more tiles than SMs
    c = helpers.workload('c1', S=S, **over)
    _set_switches(monkeypatch)
    batched = _library_choice(c)
    if c['L'] <= 4:
        assert _tc_variant(c, sms)['kernel'] == 'two' and batched[0] == 'two'
        assert _library_choice(dict(c1, S=1)) == ('pair', len(_tiles(c1)))
    else:
        assert batched[0] == 'one' and batched[1] > sms       # persistent: CTAs walk more than one item
        assert _library_choice(dict(c1, S=1))[0] == 'one'
    B, H, O = c['P'] * c['N'], c['H'], c['O']
    rng = np.random.default_rng(7)
    acts = rng.uniform(-1, 1, (S, c['N'], H, c['A'])).astype(np.float32)
    eps = rng.standard_normal((S, H, B, O), dtype=np.float32)
    states = np.asarray(c['state'], np.float32).reshape(S, O)
    for draws in ('external', 'philox'):
        e, seed, it = (eps, 0, 0) if draws == 'external' else (None, SEED64, 3)
        _set_switches(monkeypatch)
        whole = _rollout(c, acts, e, sampling, seed, it)
        assert all(np.all(np.isfinite(x)) for x in (whole[0], whole[2]))
        # the Philox counters hold the state index: a state alone is state 0, so only state 0 draws the same noise
        for s in ((0, S - 1) if draws == 'external' else (0,)):
            one = dict(c, S=1, state=states[s])
            ea = e[s:s + 1] if e is not None else None
            for switches in ((), ('SIMBA_B200_NO_PAIR',)):
                _set_switches(monkeypatch, *switches)
                got = _rollout(one, acts[s:s + 1], ea, sampling, seed, it)
                for x, y in zip(whole, got):
                    assert np.array_equal(x[s], y[0]), (draws, s, switches)
        _set_switches(monkeypatch)
