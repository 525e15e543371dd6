"""Kernel variants the host selects by shape, each held to a reference it must equal.

`simba_planner_create` picks the two-tile persistent rollout (and splits its last round) when there are more
tiles than SMs, the two-CTA pair kernel for few tiles, and the trainer picks 4-, 8- or 16-row chain tiles from
the batch. Production shapes (C4, C3, batches above 128 rows) run these variants; the other tests mostly run the
small ones. The rollout tests restate the host's choice in Python, which picks shapes without a planner per
candidate and documents the rule, and ask the library (simba_planner_rollout_kernel) whether the kernel and the
number of work items they claim to test are the ones it runs, so no test can pass because the host took a
different path.

  A  two-tile rollout (more items than SMs, split tail, padding tiles): per-row outputs bit-identical to
     the same rows through the pair kernel, one state at a time, and with the tail split switched off
  B  batched plans whose states exit early at different iterations == per-state plans, bit for bit;
     SIMBA_B200_NO_TAIL_SPLIT / NO_PDL / NO_FUSE change nothing
  C  the bf16 kernels' own Philox noise against oracle/philox.py's counter contract, row by row, with
     wrong-counter controls that must come out at least 10x worse
  D  trainer steps with 8- and 16-row chain tiles against oracle/train_oracle.py
"""
import ctypes as C

import numpy as np
import pytest

from oracle import philox
from oracle import simba_oracle as so
from oracle import train_oracle as T
from tests import helpers
from tests.test_gpu_kernels import _oracle_rows, dev, P

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

SWITCHES = ('SIMBA_B200_NO_PAIR', 'SIMBA_B200_NO_FUSE', 'SIMBA_B200_NO_PDL', 'SIMBA_B200_NO_TAIL_SPLIT')
SEED64 = 0x1234_5678_9ABC_DEF1            # both Philox key words non-zero


# ---- the host's kernel choices, restated ----------------------------------------------------------------
def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _tiles(c, group=1, rows=128):
    """build_tiles (csrc/api.cu): each member's S * rows_per_state rows (tf.split map, one rank: P*N/E rows
    per state) cut into 128-row tiles (kTcTileRows; the fp32 kernel: 32), the run padded with empty tiles to
    a multiple of `group`. -> [(member, k0, count)]"""
    m = c['P'] * c['N'] // c['E']
    tiles = []
    for e in range(c['E']):
        total = c['S'] * m
        tiles += [(e, k0, min(rows, total - k0)) for k0 in range(0, total, rows)]
        while len(tiles) % group:
            tiles.append((e, 0, 0))
    return tiles


def _tc_variant(c, sms, tail_split=True):
    """choose_rollout + split_tail_items (csrc/api.cu) for units <= 128 at most four layers (where
    rollout_tc_two_tiles_fit and rollout_tc_pair_fits hold with one constrained lidar) -> dict:
    kernel 'two' / 'pair' / 'one', items (work items of the launch), split (the tail split fired),
    pad_in_tail (an empty padding tile sat in the round that was split)."""
    assert c['U'] <= 128 and c['L'] <= 4
    tiles = _tiles(c)
    if len(tiles) <= sms:
        return dict(kernel='pair' if 2 * len(tiles) <= sms else 'one', items=len(tiles), split=False,
                    pad_in_tail=False)
    tiles = _tiles(c, 2)
    n = len(tiles) // 2
    out = dict(kernel='two', items=n, split=False, pad_in_tail=False)
    if not tail_split or n <= sms:
        return out
    last = n - sms * (-(-n // sms) - 1)
    if 2 * last > sms:
        return out
    tail = tiles[-2 * last:]
    live = sum(1 for t in tail if t[2] > 0)
    out.update(items=n - last + live, split=True, pad_in_tail=live < len(tail))
    return out


def _pick_S(c, want, start, tail_split=True):
    """The smallest S >= start for which the restated host choice satisfies want(variant); skip if the
    device's SM count allows none within reach."""
    sms = _sms()
    for S in range(start, start + 96):
        v = _tc_variant(dict(c, S=S), sms, tail_split)
        if want(v):
            switches = () if tail_split else ('SIMBA_B200_NO_TAIL_SPLIT',)
            assert _library_choice(dict(c, S=S), switches=switches) == (v['kernel'], v['items']), (S, v)
            return S, v
    pytest.skip("no S in [%d, %d) produces this variant on %d SMs" % (start, start + 96, sms))


def _library_choice(c, precision='bf16', switches=()):
    """simba_planner_rollout_kernel of a fresh planner for c, created with the given diagnostic switches set
    -> (kernel: 'fp32' / 'one' / 'pair' / 'two' / 'wide', work items of one launch)."""
    from simba_b200 import _lib
    names = {_lib.ROLLOUT_FP32: 'fp32', _lib.ROLLOUT_TC_ONE_CTA: 'one', _lib.ROLLOUT_TC_PAIR: 'pair',
             _lib.ROLLOUT_TC_TWO_TILE: 'two', _lib.ROLLOUT_TC_WIDE: 'wide'}
    kernel, items = C.c_int32(-1), C.c_int32(-1)
    with pytest.MonkeyPatch.context() as mp:
        _set_switches(mp, *switches)
        pol = helpers.cuda_policy(c, 'penalty', precision=precision)       # owns the planner handle
        _lib.check(_lib.load().simba_planner_rollout_kernel(pol._ensure_planner(), C.byref(kernel), C.byref(items)))
    return names[kernel.value], items.value


def _chain_tile_rows(E, rows):
    """chain_tile_rows (csrc/trainer.cu): the smallest row tile that keeps E x row tiles within 160 CTAs."""
    for R in (4, 8):
        if E * -(-rows // R) <= 160:
            return R
    return 16


# ---- small helpers ----------------------------------------------------------------------------------------
def _set_switches(monkeypatch, *on):
    for name in SWITCHES:
        if name in on:
            monkeypatch.setenv(name, '1')
        else:
            monkeypatch.delenv(name, raising=False)


def _rollout(c, precision, acts, eps, seed=0, it=0):
    """One simba_rollout_score call on a fresh planner for c['S'] states: acts [S, N, H, A], eps
    [S, H, P*N, O] or None (device Philox) -> (return, cost mask, cost sum), each [S, P*N]."""
    from simba_b200 import _lib
    lib = _lib.load()
    pol = helpers.cuda_policy(c, 'penalty', precision=precision)
    pl = pol._ensure_planner()
    S, B = c['S'], c['P'] * c['N']
    ret = torch.full((S * B,), np.nan, dtype=torch.float32, device='cuda')
    mask = torch.full((S * B,), -1, dtype=torch.int64, device='cuda')
    csum = torch.full((S * B,), np.nan, dtype=torch.float32, device='cuda')
    d_state = dev(np.asarray(c['state'], np.float32).reshape(S, c['O']))
    d_acts = dev(acts)
    d_eps = dev(eps) if eps is not None else None
    _lib.check(lib.simba_rollout_score(pl, P(d_state), P(d_acts), P(d_eps), seed, it, None, P(ret), P(mask),
                                       P(csum), None))
    torch.cuda.synchronize()
    return tuple(x.cpu().numpy().reshape(S, B) for x in (ret, mask, csum))


def _states(c):
    return np.asarray(c['state'], np.float32).reshape(c['S'], c['O'])


def _one_state(c, s):
    c1 = dict(c, S=1)
    c1['state'] = _states(c)[s]
    return c1


def _assert_rows_close_to_oracle(c, got, acts, eps):
    """The bf16 tolerance of tests/test_gpu_tc.py: mean |d return| < 1e-2, mask agreement > 1 - 0.002 H,
    per-candidate mean return within 2e-2."""
    traj, cum0, mask0, _ = _oracle_rows(c, helpers.oracle_planner(c, 'penalty'), acts, eps, 'penalty')
    ret, mask, _ = got
    assert np.abs(ret - cum0).mean() < 1e-2
    assert (mask.view(np.uint64) == mask0).mean() > 1.0 - 0.002 * c['H']
    cand = np.abs(ret.reshape(c['P'], c['N']).mean(0) - cum0.reshape(c['P'], c['N']).mean(0))
    assert cand.max() < 2e-2


# ---- the rollout kernels of the benchmark's shapes -----------------------------------------------------------
BENCH_SHAPES = {              # (workload, overrides, precision, kernel)
    'c1': ('c1', dict(), 'bf16', 'pair'),                 # the headline plan: one state, 25 tiles
    'c1-16-states': ('c1', dict(S=16), 'bf16', 'two'),    # 375 tiles, the last round split
    'c4': ('c4', dict(), 'bf16', 'two'),                  # 1024 states per call
    'c5': ('c5', dict(), 'bf16', 'wide'),
    'c1-fp32': ('c1', dict(), 'fp32', 'fp32'),
}


@pytest.mark.parametrize("shape", list(BENCH_SHAPES))
def test_benchmark_shapes_run_the_expected_rollout_kernel(shape):
    cfg, over, precision, kernel = BENCH_SHAPES[shape]
    c = helpers.workload(cfg, **over)
    got = _library_choice(c, precision)
    if kernel == 'fp32':
        assert got == ('fp32', len(_tiles(c, rows=32)))
    elif kernel == 'wide':
        assert got == ('wide', len(_tiles(c)))
    else:
        v = _tc_variant(c, _sms())
        assert v['kernel'] == kernel and got == (kernel, v['items'])
        if shape == 'c1-16-states':
            assert v['split'] and got[1] > _library_choice(c, switches=('SIMBA_B200_NO_TAIL_SPLIT',))[1]


# ---- A: two-tile persistent rollout, per row, bit for bit ---------------------------------------------------
CASES_A = {
    # C1 dims: more work items than SMs, and the last round split into single tiles (375 tiles at S = 16)
    'c1-split': (dict(), lambda v: v['kernel'] == 'two' and v['items'] > _sms() and v['split'], 16),
    # more items than SMs, last round too full to split (235 items at S = 20)
    'c1-no-split': (dict(), lambda v: v['kernel'] == 'two' and v['items'] > _sms() and not v['split'], 20),
    # three members with an odd tile run each: padding tiles, one of them in the split round
    'three-members': (dict(E=3), lambda v: v['kernel'] == 'two' and v['split'] and v['pad_in_tail'], 8),
}


@pytest.mark.parametrize("case", list(CASES_A))
def test_two_tile_rollout_rows_equal_pair_kernel_rows(case, monkeypatch):
    """The persistent two-tile kernel's item loop, weight re-staging on a member change, padding tiles and
    split tail against the pair kernel on each state alone (which the suite holds to the one-CTA kernel
    and to the oracle): ret, cost mask and cost sum bit-identical per row, also without the tail split."""
    over, want, start = CASES_A[case]
    S, v = _pick_S(helpers.workload('c1', **over), want, start)
    c = helpers.workload('c1', S=S, **over)
    sms = _sms()
    one, whole = _tc_variant(dict(c, S=1), sms), _tc_variant(c, sms, tail_split=False)
    assert one['kernel'] == 'pair' and whole['kernel'] == 'two'
    assert _library_choice(dict(c, S=1)) == ('pair', one['items'])
    assert _library_choice(c, switches=('SIMBA_B200_NO_TAIL_SPLIT',)) == ('two', whole['items'])
    print("%s: S=%d %s" % (case, S, v))
    B, H, O = c['P'] * c['N'], c['H'], c['O']
    rng = np.random.default_rng(21)
    acts = rng.uniform(-1, 1, (S, c['N'], H, c['A'])).astype(np.float32)
    eps = rng.standard_normal((S, H, B, O), dtype=np.float32)
    _set_switches(monkeypatch)
    base = _rollout(c, 'bf16', acts, eps)
    assert all(np.all(np.isfinite(x)) for x in (base[0], base[2]))
    _set_switches(monkeypatch, 'SIMBA_B200_NO_TAIL_SPLIT')
    whole = _rollout(c, 'bf16', acts, eps)
    _set_switches(monkeypatch)
    for x, y in zip(base, whole):
        assert np.array_equal(x, y)
    for s in range(S):
        one = _rollout(_one_state(c, s), 'bf16', acts[s:s + 1], eps[s:s + 1])
        for x, y in zip(base, one):
            assert np.array_equal(x[s], y[0]), s
    for s in (0, S - 1):
        _assert_rows_close_to_oracle(_one_state(c, s), tuple(x[s] for x in base), acts[s], eps[s])
    # Philox mode: the split and the unsplit item lists draw the same noise for the same rows
    ph = _rollout(c, 'bf16', acts, None, SEED64, 3)
    _set_switches(monkeypatch, 'SIMBA_B200_NO_TAIL_SPLIT')
    ph_whole = _rollout(c, 'bf16', acts, None, SEED64, 3)
    for x, y in zip(ph, ph_whole):
        assert np.array_equal(x, y)
    assert not np.array_equal(ph[0], base[0])


# ---- B: batched plans with per-state early exit == per-state plans --------------------------------------
def _plan(c, monkeypatch, switches=(), draws=None, seed=None, **kw):
    from simba_b200 import _lib
    _set_switches(monkeypatch, *switches)
    pol = helpers.cuda_policy(c, 'penalty', precision='bf16', **kw)
    if draws is not None:
        pol.set_external_draws(*draws)
    a, s = pol.do_generate_action(_states(c), seed=seed)
    S = c['S']
    out = dict(action=np.asarray(a).reshape(S, -1), score=np.asarray(s).reshape(S),
               iters=np.asarray(pol.iterations_run).reshape(S).copy(),
               mu=pol.buffer(_lib.BUF_MU).cpu().numpy().reshape(S, -1),
               sigma=pol.buffer(_lib.BUF_SIGMA).cpu().numpy().reshape(S, -1),
               elite=pol.buffer(_lib.BUF_ELITE, torch.int32).cpu().numpy().reshape(S, -1))
    _set_switches(monkeypatch)
    return out


def _assert_plans_equal(a, b, s=None):
    for k in a:
        x = a[k] if s is None else a[k][s:s + 1]
        assert np.array_equal(x, b[k]), (k, s)


def _assert_per_state_plans_equal(c, batched, draws, monkeypatch, **kw):
    z, eps, zf = draws
    for s in range(c['S']):
        one = _plan(_one_state(c, s), monkeypatch, draws=(z[:, s:s + 1], eps[:, s:s + 1], zf[s:s + 1]), **kw)
        _assert_plans_equal(batched, one, s)


def test_batched_two_tile_plans_with_early_exit_equal_per_state_plans(monkeypatch):
    """C1 dims, 16 states (two-tile kernel, split tail) with a stddev threshold that stops some states after
    the first iteration and others later: items whose states have all stopped are skipped (tile_active),
    members change around them. Every state's action, score, iteration count, final mean / stddev and elite
    set equal a one-state plan on the same draws, bit for bit; the diagnostic switches change nothing."""
    from simba_b200 import synthetic
    S, v = _pick_S(helpers.workload('c1', H=8, I=4),
                   lambda v: v['kernel'] == 'two' and v['items'] > _sms() and v['split'], 16)
    c = helpers.workload('c1', S=S, H=8, I=4)
    draws = synthetic.make_draws(c['I'], S, c['N'], c['H'], c['A'], c['P'], c['O'], seed=5)
    thr = 0.67            # between the first-iteration stddev means of these states (C1 dims, H = 8)
    base = _plan(c, monkeypatch, draws=draws, stddev_threshold=thr)
    print("S=%d %s iterations %s" % (S, v, base['iters']))
    assert base['iters'].min() == 1 and len(set(base['iters'].tolist())) >= 2
    assert np.all(np.isfinite(base['score']))
    _assert_per_state_plans_equal(c, base, draws, monkeypatch, stddev_threshold=thr)
    for sw in ('SIMBA_B200_NO_TAIL_SPLIT', 'SIMBA_B200_NO_PDL', 'SIMBA_B200_NO_FUSE'):
        _assert_plans_equal(base, _plan(c, monkeypatch, (sw,), draws=draws, stddev_threshold=thr))


@pytest.mark.parametrize("cfg", ['c1', 'wide'])
def test_plans_without_programmatic_dependent_launch_are_bit_identical(cfg, monkeypatch):
    """Production mode (device Philox, CUDA graph): a dependent kernel that read anything before its
    griddepcontrol.wait would read it the same way every replay, so only the plan without programmatic
    dependent launches (SIMBA_B200_NO_PDL=1) can show it. C1: the pair kernel's late wait; wide: the
    streaming kernel over three states."""
    c = helpers.workload('c1') if cfg == 'c1' else helpers.workload('tiny', U=400, L=2, S=3)
    if cfg == 'c1':
        v = _tc_variant(c, _sms())
        assert v['kernel'] == 'pair' and _library_choice(c) == ('pair', v['items'])
    else:
        assert _library_choice(c) == ('wide', len(_tiles(c)))
    base = _plan(c, monkeypatch, seed=SEED64)
    plain = _plan(c, monkeypatch, ('SIMBA_B200_NO_PDL',), seed=SEED64)
    _assert_plans_equal(base, plain)
    assert not np.array_equal(base['action'], _plan(c, monkeypatch, seed=SEED64 + 1)['action'])


def test_wide_batched_plans_equal_per_state_plans(monkeypatch):
    """The wide kernel's tiles straddle states; on external draws each state's plan equals a one-state plan."""
    from simba_b200 import synthetic
    c = helpers.workload('tiny', U=400, L=2, S=3)
    draws = synthetic.make_draws(c['I'], 3, c['N'], c['H'], c['A'], c['P'], c['O'], seed=6)
    tiles = _tiles(c)
    assert _library_choice(c) == ('wide', len(tiles))
    assert any(k0 // (c['P'] * c['N'] // c['E']) != (k0 + n - 1) // (c['P'] * c['N'] // c['E'])
               for _, k0, n in tiles)                         # a tile holds rows of two states
    base = _plan(c, monkeypatch, draws=draws)
    _assert_per_state_plans_equal(c, base, draws, monkeypatch)


# ---- C: in-kernel noise vs the Philox counter contract --------------------------------------------------
# (cfg, overrides, sensors, switches, the noise code path it reaches)
PATHS_C = {
    # one item per cluster (C1: 50 tiles for two states): Q = 4, one Philox block per thread and step,
    # its ten rounds after an even layer and Box-Muller after the next (rollout_tc.cu, latency variant)
    'pair-latency': ('c1', dict(S=2), None, ()),
    # one-CTA kernel (NO_PAIR), two blocks per thread and step, L < 4: make_noise, one block per layer
    'one-cta-L2': ('tiny', dict(S=2, L=2), None, ('SIMBA_B200_NO_PAIR',)),
    # L = 1: the second block is drawn after the last layer
    'one-cta-L1': ('tiny', dict(S=2, L=1), None, ('SIMBA_B200_NO_PAIR',)),
    # more than 148 tiles: the two-tile kernel, four blocks per thread parked in shared memory
    'two-tile': ('c1', dict(), None, ()),
    # units 400: rollout_tc_wide.cu
    'wide': ('tiny', dict(S=2, U=400, L=2), None, ()),
    # O = 22 (simple lidar): the last block of a row is masked (mask_noise8), 75 tiles: one-CTA kernel
    'obs22': ('shipped', dict(S=2, N=100), 'simple', ()),
}


def _path_workload(path):
    from simba_b200 import synthetic
    cfg, over, sensors, switches = PATHS_C[path]
    over = dict(over)
    if path == 'two-tile':                      # the smallest S above 148 tiles (7 at C1)
        over['S'], _ = _pick_S(helpers.workload('c1'), lambda v: v['kernel'] == 'two', 2)
    c = helpers.workload(cfg, sensors=synthetic.POINTSIMPLEGOAL1_SENSORS if sensors else None, **over)
    if c['U'] <= 128:
        v = _tc_variant(c, _sms())
        expect = {'pair-latency': 'pair', 'two-tile': 'two'}.get(path, 'one')
        got = 'one' if (v['kernel'] == 'pair' and switches) else v['kernel']
        assert got == expect, (path, v)
        assert _library_choice(c, switches=switches) == (got, v['items']), (path, v)
    else:
        assert _library_choice(c, switches=switches) == ('wide', len(_tiles(c))), path
    assert c['S'] >= 2
    return c, switches


def _contract_eps(c, seed, it, rows=None, state=None, t0=0):
    """eps [S, H, P*N, O] of oracle/philox.noise_normals; the keyword arguments move one counter field."""
    B = c['P'] * c['N']
    rows = np.arange(B) if rows is None else rows
    out = np.empty((c['S'], c['H'], B, c['O']), np.float32)
    for s in range(c['S']):
        si = s if state is None else state(s)
        out[s] = philox.noise_normals(seed, it, c['H'] + t0, rows, c['O'], state_index=si)[t0:]
    return out


def _controls(c, seed, it):
    B, N, P_ = c['P'] * c['N'], c['N'], c['P']
    r = np.arange(B)
    return {
        'iteration+1': lambda: _contract_eps(c, seed, it + 1),
        'iteration-1': lambda: _contract_eps(c, seed, it - 1),
        'other state': lambda: _contract_eps(c, seed, it, state=lambda s: (s + 1) % c['S']),
        't+1': lambda: _contract_eps(c, seed, it, t0=1),
        'rows candidate-major': lambda: _contract_eps(c, seed, it, rows=(r % N) * P_ + r // N),
        'rows shifted': lambda: _contract_eps(c, seed, it, rows=r + 1),
        'seed high word dropped': lambda: _contract_eps(c, seed & 0xFFFFFFFF, it),
    }


# MUFU normals (device) and the accurate contract normals, both rounded to bf16, differ in a few draws, which
# moves a few rows' returns slightly. Measured on a B200 (148 SMs, 1000 W) at these shapes: mean |d return|
# 0 to 4.3e-7, masks and cost sums identical in every row; every wrong-counter control >= 0.061 (t + 1),
# about 0.2 for the others, i.e. >= 1.5e5 times the contract's difference. Pinned about 10x above.
NOISE_BOUNDS = dict(mean_dret=5e-6, mask_same=0.999, csum_same=0.999)


@pytest.mark.parametrize("path", list(PATHS_C))
def test_bf16_device_noise_follows_the_philox_contract(path, monkeypatch):
    c, switches = _path_workload(path)
    it = 3
    rng = np.random.default_rng(31)
    acts = rng.uniform(-1, 1, (c['S'], c['N'], c['H'], c['A'])).astype(np.float32)
    _set_switches(monkeypatch, *switches)
    dev_rows = _rollout(c, 'bf16', acts, None, SEED64, it)

    def compare(eps):
        ret, mask, csum = _rollout(c, 'bf16', acts, eps)
        return (np.abs(ret - dev_rows[0]).mean(), (mask == dev_rows[1]).mean(), (csum == dev_rows[2]).mean())

    good = compare(_contract_eps(c, SEED64, it))
    print("%s S=%d: contract mean|dret| %.3g, masks identical %.4f, cost sums identical %.4f"
          % (path, c['S'], *good))
    assert np.all(np.isfinite(dev_rows[0]))
    assert good[0] <= NOISE_BOUNDS['mean_dret']
    assert good[1] >= NOISE_BOUNDS['mask_same'] and good[2] >= NOISE_BOUNDS['csum_same']
    for name, make in _controls(c, SEED64, it).items():
        bad = compare(make())
        print("  control %-22s mean|dret| %.3g  ratio %.3g" % (name, bad[0], bad[0] / max(good[0], 1e-12)))
        assert bad[0] >= 10 * good[0] and bad[0] > 0, name


def _fragile(c, traj):
    """Rows whose goal / hazard decision sits within 1e-4 of its threshold in the oracle (as in
    test_rollout_score_rows_match_oracle)."""
    sc = so.Scorer(None, c['table'])
    frag = np.zeros(traj.shape[0], bool)
    for t in range(c['H'] + 1):
        frag |= np.abs(sc.goal_distance_metric(traj[:, t]) - np.float32(0.24)) < 1e-4
        frag |= np.abs(sc.closest_distance(traj[:, t][:, c['table']['hazards_lidar']]) - np.float32(0.2)) < 1e-4
    return frag


@pytest.mark.parametrize("path", [p for p in PATHS_C if p != 'two-tile'])
def test_fp32_device_noise_follows_the_philox_contract(path, monkeypatch):
    """The fp32 kernel's accurate Philox normals at the same shapes, 64-bit seed, iteration 3, several
    states: its rows equal the oracle fed with the contract normals within 1e-4 on non-fragile rows."""
    c, _ = _path_workload(path)
    it = 3
    rng = np.random.default_rng(32)
    acts = rng.uniform(-1, 1, (c['S'], c['N'], c['H'], c['A'])).astype(np.float32)
    _set_switches(monkeypatch)
    ret, mask, csum = _rollout(c, 'fp32', acts, None, SEED64, it)
    eps = _contract_eps(c, SEED64, it)
    for s in range(c['S']):
        cs = _one_state(c, s)
        traj, cum0, mask0, csum0 = _oracle_rows(cs, helpers.oracle_planner(cs, 'penalty'), acts[s], eps[s], 'penalty')
        ok = ~_fragile(cs, traj)
        assert ok.mean() > 0.98
        assert np.allclose(ret[s][ok], cum0[ok], rtol=1e-4, atol=2e-5), s
        assert np.array_equal(mask[s].view(np.uint64)[ok], mask0[ok]), s
        assert np.array_equal(csum[s][ok], csum0[ok]), s


def test_sample_actions_philox_several_states_64bit_seed():
    from simba_b200 import _lib
    lib = _lib.load()
    c = helpers.workload('c1', S=3)
    pol = helpers.cuda_policy(c, 'penalty')           # owns the planner handle: keep it alive
    pl = pol._ensure_planner()
    S, N, H, A = 3, c['N'], c['H'], c['A']
    rng = np.random.default_rng(33)
    mu = rng.uniform(-0.5, 0.5, (S, H, A)).astype(np.float32)
    sg = rng.uniform(0.1, 1.0, (S, H, A)).astype(np.float32)
    out = torch.empty((S, N, H, A), dtype=torch.float32, device='cuda')
    d_mu, d_sg = dev(mu), dev(sg)
    _lib.check(lib.simba_sample_actions(pl, P(d_mu), P(d_sg), None, SEED64, 7, None, P(out), None))
    torch.cuda.synchronize()
    got = out.cpu().numpy()
    for s in range(S):
        zz = philox.action_normals(SEED64, 7, N, H, A, state_index=s)
        ref = np.minimum(np.maximum(zz * sg[s] + mu[s], np.float32(-1)), np.float32(1))
        assert np.max(np.abs(got[s] - ref)) < 5e-6, s


# ---- D: trainer with 8- and 16-row chain tiles ----------------------------------------------------------
def _ensemble(n_in, n_out, E, B, L, U, lr=0.00025, steps=5000, dropout=0.0, seed=0):
    from simba_b200.models import MlpEnsemble
    return MlpEnsemble(n_in, n_out, E, batch_size=B, learning_rate=lr, learning_rate_schedule=False,
                       training_steps=steps, mlp_params=dict(n_layers=L, units=U, dropout_rate=dropout), seed=seed)


def _oracle(ens, dropout=0.0):
    return T.EnsembleTrainer([m.get_weights() for m in ens.ensemble], batch_size=ens.batch_size,
                             learning_rate=ens.learning_rate, learning_rate_schedule=False,
                             training_steps=ens.training_steps, dropout_rate=dropout, dropout_seed=ens.dropout_seed)


def _relu_margin(ora, x):
    """Smallest |pre-activation| of any hidden unit in the oracle's forward pass (with its dropout masks)."""
    m = np.inf
    for e, net in enumerate(ora.nets):
        h = x[e]
        for l in range(net.n_layers):
            z = h @ net.arrays[2 * l] + net.arrays[2 * l + 1]
            m = min(m, float(np.abs(z).min()))
            h = np.maximum(z, 0)
            if ora.dropout_rate > 0:
                keep = philox.dropout_keep(ora.dropout_seed, ora.optimizer.iterations, e, l, h.shape[0], h.shape[1],
                                           ora.dropout_rate)
                h = h * keep / np.float32(1 - ora.dropout_rate)
    return m


def _clear_batch(ora, rng, E, rows, n_in, n_out, scale=1.0):
    """A batch none of whose hidden pre-activations lies within 1e-6 of the ReLU kink: there two correct
    fp32 summation orders may disagree on the mask, and a whole unit's gradient then differs by a row's
    share. At 512 rows x 4 layers x 128 units a batch holds a few such values in expectation."""
    for _ in range(200):
        x = rng.uniform(0, 1, (E, rows, n_in)).astype(np.float32)
        y = (rng.normal(0, 0.1, (E, rows, n_out)) * scale).astype(np.float32)
        if _relu_margin(ora, x) > 1e-6:
            return x, y
    raise AssertionError("no batch clear of the ReLU kink")


def _assert_state_matches(ens, ora, E, L, grad_tol, m_tol, w_tol):
    n_var = 2 * L + 4
    for e in range(E):
        for got, ref in zip(ens.trainer_arrays('grads', e), ora.last_grads[e * n_var:(e + 1) * n_var]):
            np.testing.assert_allclose(got, ref, **grad_tol)
        for got, ref in zip(ens.trainer_arrays('m', e), ora.optimizer.m[e * n_var:(e + 1) * n_var]):
            np.testing.assert_allclose(got, ref, **m_tol)
        for got, ref in zip(ens.trainer_arrays('weights', e), ora.nets[e].arrays):
            np.testing.assert_allclose(got, ref, **w_tol)


# (n_in, n_out, E, batch_size, rows, L, U, chain tile rows)
SHAPES_D = [
    (12, 10, 5, 128, 128, 2, 40, 4),            # the exact boundaries of chain_tile_rows at E = 5
    (12, 10, 5, 129, 129, 2, 40, 8),
    (12, 10, 5, 256, 256, 2, 40, 8),
    (12, 10, 5, 257, 257, 2, 40, 16),
    (62, 60, 5, 512, 512, 4, 128, 16),          # C1 dims: eight 64-row chunks in the update kernel
    (9, 7, 2, 400, 400, 2, 130, 8),             # unaligned: U = 130, 2 O = 14 not a multiple of 4
    (20, 18, 3, 500, 500, 3, 200, 16),
    (12, 10, 5, 512, 300, 2, 40, 16),           # fewer rows than batch_size: R follows the rows
]


@pytest.mark.parametrize('shape', SHAPES_D)
def test_one_step_with_wide_chain_tiles_matches_oracle(shape):
    n_in, n_out, E, B, rows, L, U, R = shape
    assert _chain_tile_rows(E, rows) == R
    ens = _ensemble(n_in, n_out, E, B, L, U)
    ora = _oracle(ens)
    x, y = _clear_batch(ora, np.random.default_rng(41), E, rows, n_in, n_out)
    loss, want = float(ens.training_step(x, y)), float(ora.training_step(x, y))
    assert loss == pytest.approx(want, rel=1e-4)
    _assert_state_matches(ens, ora, E, L, dict(rtol=1e-4, atol=1e-7), dict(rtol=1e-4, atol=1e-8),
                          dict(rtol=1e-4, atol=ens.learning_rate * 0.02))
    assert ens.iterations == 1


def test_several_steps_with_wide_chain_tiles_and_clipvalue():
    """Loss, gradients, Adam m and weights over six steps at R = 16; the first two steps' targets are large
    enough that gradients pass clipvalue 1.0."""
    n_in, n_out, E, B, L, U = 12, 10, 5, 300, 2, 40
    assert _chain_tile_rows(E, B) == 16
    ens = _ensemble(n_in, n_out, E, B, L, U, lr=1e-3)
    ora = _oracle(ens)
    rng = np.random.default_rng(42)
    clipped = False
    for s in range(6):
        x, y = _clear_batch(ora, rng, E, B, n_in, n_out, scale=300.0 if s < 2 else 1.0)
        got, want = float(ens.training_step(x, y)), float(ora.training_step(x, y))
        clipped |= any(np.abs(g).max() > 1.0 for g in ora.last_grads)
        assert got == pytest.approx(want, rel=2e-4), s
    assert clipped
    _assert_state_matches(ens, ora, E, L, dict(rtol=2e-3, atol=2e-6), dict(rtol=2e-3, atol=2e-7),
                          dict(rtol=0, atol=4e-3))
    assert ens.iterations == 6


@pytest.mark.parametrize('E', [5, 6])
def test_fit_with_uneven_batches_at_wide_chain_tiles(E):
    """fit() (graph replay, gathered batches) at batch_size 256: np.array_split gives 251 / 250-row batches,
    the row tile is chosen from batch_size (8 rows at E = 5, 16 at E = 6)."""
    n_in, n_out, B, L, U, steps = 12, 10, 256, 2, 40, 12
    assert _chain_tile_rows(E, B) == {5: 8, 6: 16}[E]
    ens = _ensemble(n_in, n_out, E, B, L, U, lr=5e-4, steps=steps)
    ens.validation_split = 0.0
    ora = _oracle(ens)
    rng = np.random.default_rng(43)
    n = 1001
    x = rng.uniform(0, 1, (n, n_in)).astype(np.float32)
    y = rng.normal(0, 0.1, (n, n_out)).astype(np.float32)
    np.random.seed(12)
    losses = ens.fit(x, y)
    np.random.seed(12)
    train_idx, _ = ens._split_indices(n)
    index, rows = ens.batch_schedule(n, steps)
    assert sorted(set(rows.tolist())) == [250, 251]
    want = ora.fit_batches(x, y, [train_idx[index[s, :, :rows[s]]] for s in range(steps)])
    np.testing.assert_allclose(losses, want, rtol=2e-4)
    for e in range(E):
        for got, ref in zip(ens.ensemble[e].get_weights(), ora.nets[e].arrays):
            np.testing.assert_allclose(got, ref, rtol=0, atol=4 * 5e-4)
    assert ens.iterations == steps


def test_dropout_steps_with_sixteen_row_chain_tiles():
    n_in, n_out, E, B, L, U, rate = 20, 18, 3, 500, 3, 200, 0.25
    assert _chain_tile_rows(E, B) == 16
    ens = _ensemble(n_in, n_out, E, B, L, U, lr=1e-3, dropout=rate, seed=7)
    ora = _oracle(ens, dropout=rate)
    rng = np.random.default_rng(44)
    for s in range(3):
        x, y = _clear_batch(ora, rng, E, B, n_in, n_out)
        got, want = float(ens.training_step(x, y)), float(ora.training_step(x, y))
        assert got == pytest.approx(want, rel=2e-4, abs=1e-6), s
    _assert_state_matches(ens, ora, E, L, dict(rtol=2e-3, atol=2e-6), dict(rtol=2e-3, atol=2e-7),
                          dict(rtol=0, atol=1.2e-2))


def test_validation_step_with_eight_row_chain_tiles():
    n_in, n_out, E, L, U, rows = 12, 10, 3, 2, 40, 300
    assert _chain_tile_rows(E, rows) == 8
    ens = _ensemble(n_in, n_out, E, 16, L, U)
    ora = _oracle(ens)
    rng = np.random.default_rng(45)
    x = rng.uniform(0, 1, (rows, n_in)).astype(np.float32)
    y = rng.normal(0, 0.1, (rows, n_out)).astype(np.float32)
    assert float(ens.validation_step(x, y)) == pytest.approx(float(ora.validation_step(x, y)), rel=1e-4)
