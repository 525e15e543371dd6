"""bf16 tcgen05 rollouts for observations wider than 60 dims: rollout_tc_wide.cu's 128-state-column variant
(SIMBA_ROLLOUT_TC_WIDE_OBS), which the host selects only for bf16 shapes every other tcgen05 kernel rejects
(obs_dim + act_dim + 2 <= 128, obs_dim <= 124, act_dim <= 4, units <= 384).

  1  kernel choice: the shapes that now run report the new kernel with one work item per tile; the benchmark
     shapes keep theirs; shapes beyond its limits are still rejected with SIMBA_ERR_UNSUPPORTED
  2  rows against the oracle on external draws, at tests/test_gpu_tc.py's bf16 tolerances
  3  the kernel's own Philox noise against oracle/philox.py's counter contract (with wrong-counter controls)
  4  whole plans, bf16 against fp32 on the same draws
  5  bit-identical checks: batched vs per-state plans with early exit, the diagnostic switches, re-committed
     weights, and (two GPUs) the population-sharded plan
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from tests import helpers
from tests.test_gpu_dispatch_variants import (NOISE_BOUNDS, SEED64, _contract_eps, _controls, _one_state,
                                              _rollout, _set_switches, _tiles)
from tests.test_gpu_kernels import _oracle_rows, dev, P

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# Sensor layouts (offsets by sorted key, as safety_gym.py lays them out). Goal + four constrained lidar classes at
# the default 16 bins is 92 dims: accelerometer [0, 3), goal [3, 19), gremlins [19, 35) (straddles the 32-dim
# slice of one epilogue thread), gyro, hazards [38, 54), magnetometer, pillars [57, 73) (straddles dim 64: layer
# 0's second K atom), vases [73, 89), velocimeter [89, 92).
ROBOT = dict(accelerometer=3, gyro=3, magnetometer=3, velocimeter=3)
GOAL4 = dict(ROBOT, goal_lidar=16, gremlins_lidar=16, hazards_lidar=16, pillars_lidar=16, vases_lidar=16)
GOAL3 = dict(ROBOT, goal_lidar=16, hazards_lidar=16, pillars_lidar=16, vases_lidar=16)           # 76
SENSORS = {
    61: dict(ROBOT, goal_lidar=16, hazards_lidar=16, vases_lidar=16, velocimeter=4),
    63: dict(ROBOT, goal_lidar=16, hazards_lidar=16, vases_lidar=16, velocimeter=6),   # a_t at dims 63, 64
    76: GOAL3,
    92: GOAL4,
    123: dict(GOAL4, joints=31),                                                       # A = 3: O + A + 2 = 128
    124: dict(GOAL4, joints=32),                                                       # O + A + 2 = 128
    125: dict(GOAL4, joints=33),          # A = 1: O + A + 2 = 128, but a_t's four state columns would pass 128
    126: dict(GOAL4, joints=34),
    # goal_dist observation at index 67 (the 'aux' block sorts before it)
    'goal_dist': dict(accelerometer=3, aux=64, goal_dist=1, hazards_lidar=16, vases_lidar=16),
    60: None,                                                                          # PointGoal1
}
SCORERS = {
    'goal4': dict(constrain_vases=True, constrain_hazards=True, constrain_pillars=True, constrain_gremlins=True),
    'goal3': dict(constrain_vases=True, constrain_hazards=True, constrain_pillars=True),
    'goal_dist': dict(observe_goal_lidar=False, observe_goal_dist=True, constrain_vases=True),
}


def _workload(obs, cfg='tiny', **over):
    return helpers.workload(cfg, sensors=SENSORS[obs], **over)


def _choice(c, precision='bf16', scorer_config=None, switches=()):
    """simba_planner_rollout_kernel of a fresh planner -> (kernel constant, work items)."""
    from simba_b200 import _lib
    kernel, items = C.c_int32(-1), C.c_int32(-1)
    with pytest.MonkeyPatch.context() as mp:
        _set_switches(mp, *switches)
        pol = helpers.cuda_policy(c, 'penalty', precision=precision, scorer_config=scorer_config)
        _lib.check(_lib.load().simba_planner_rollout_kernel(pol._ensure_planner(), C.byref(kernel), C.byref(items)))
    return kernel.value, items.value


# ---- 1: kernel choice ----------------------------------------------------------------------------------------
RUNS = {                   # name: (obs, overrides, scorer)
    'o61': (61, dict(), None),
    'o76': (76, dict(), 'goal3'),
    'o92': (92, dict(), 'goal4'),
    'o124': (124, dict(), 'goal4'),
    'o124-a1': (124, dict(A=1), 'goal4'),
    'o123-a3': (123, dict(A=3), 'goal4'),
    'o92-u64': (92, dict(U=64), 'goal4'),
    'o92-u200': (92, dict(U=200), 'goal4'),
    'o92-u256': (92, dict(U=256), 'goal4'),
    'o92-u320': (92, dict(U=320), 'goal4'),
    'o60-a4-u256': (60, dict(A=4, U=256), None),
    'o92-l6': (92, dict(L=6), 'goal4'),
    'o92-u384': (92, dict(U=384, L=2), 'goal4'),
}


@pytest.mark.parametrize("name", list(RUNS))
def test_wide_observation_shapes_run_the_new_kernel(name):
    from simba_b200 import _lib
    obs, over, scorer = RUNS[name]
    for S in (1, 3):
        c = _workload(obs, S=S, **over)
        assert _choice(c, scorer_config=SCORERS.get(scorer)) == (_lib.ROLLOUT_TC_WIDE_OBS, len(_tiles(c)))
        # fp32 still runs the fp32 kernel, and NO_PAIR / NO_TAIL_SPLIT do not apply
        assert _choice(c, 'fp32')[0] == _lib.ROLLOUT_FP32
        assert _choice(c, switches=('SIMBA_B200_NO_PAIR', 'SIMBA_B200_NO_TAIL_SPLIT'),
                       scorer_config=SCORERS.get(scorer)) == (_lib.ROLLOUT_TC_WIDE_OBS, len(_tiles(c)))


@pytest.mark.parametrize("cfg,over,kernel", [
    ('c1', dict(), 'TC_PAIR'), ('c1', dict(S=16), 'TC_TWO_TILE'), ('c4', dict(), 'TC_TWO_TILE'),
    ('c5', dict(), 'TC_WIDE'), ('tiny', dict(U=256), 'TC_WIDE'), ('tiny', dict(L=5), 'TC_ONE_CTA')])
def test_shapes_that_ran_before_keep_their_kernel(cfg, over, kernel):
    from simba_b200 import _lib
    c = helpers.workload(cfg, **over)
    assert _choice(c)[0] == getattr(_lib, 'ROLLOUT_' + kernel)


@pytest.mark.parametrize("obs,over", [(126, dict()), (125, dict(A=1)), (92, dict(A=5)), (92, dict(U=400, L=2))])
def test_shapes_beyond_the_new_kernel_are_still_rejected(obs, over):
    from simba_b200 import _lib
    c = _workload(obs, **over)
    pol = helpers.cuda_policy(c, 'penalty', precision='bf16')
    with pytest.raises(_lib.SimbaError) as e:
        pol._ensure_planner()
    assert e.value.code == -6 and 'obs_dim+act_dim <= 126' in str(e.value)
    helpers.cuda_policy(c, 'penalty', precision='fp32')._ensure_planner()      # the fp32 kernel takes them


# ---- 2: rows against the oracle ----------------------------------------------------------------------------
ROWS = {                   # name: (obs, overrides, scorer, objective, sampling_propagation)
    'o61-L4': (61, dict(L=4), None, 'penalty', True),
    'o63-a2-actions-straddle-64': (63, dict(L=2), None, 'penalty', True),
    'o76-L1': (76, dict(L=1), 'goal3', 'penalty', True),
    'o92-L4-goal4': (92, dict(L=4), 'goal4', 'penalty', True),
    'o92-L6-goal4': (92, dict(L=6), 'goal4', 'penalty', True),
    'o92-L4-reward': (92, dict(L=4), 'goal4', 'reward', True),
    'o92-L4-no-sampling': (92, dict(L=4), 'goal4', 'penalty', False),
    'o92-u64': (92, dict(U=64, L=2), 'goal4', 'penalty', True),
    'o92-u200': (92, dict(U=200, L=3), 'goal4', 'penalty', True),
    'o92-u256': (92, dict(U=256, L=2), 'goal4', 'penalty', True),
    'o92-u320-L1': (92, dict(U=320, L=1), 'goal4', 'penalty', True),
    'o124-L4': (124, dict(L=4), 'goal4', 'penalty', True),
    'o124-a1': (124, dict(A=1, L=2), 'goal4', 'penalty', True),
    'o123-a3': (123, dict(A=3, L=2), 'goal4', 'penalty', True),
    'o60-a4-u256': (60, dict(A=4, U=256, L=2), None, 'penalty', True),
    'goal-dist-67': ('goal_dist', dict(L=2), 'goal_dist', 'penalty', True),
}


@pytest.mark.parametrize("name", list(ROWS))
def test_rows_close_to_oracle(name):
    from simba_b200 import _lib
    obs, over, scorer, objective, sampling = ROWS[name]
    lib = _lib.load()
    c = _workload(obs, **over)
    cfg = SCORERS.get(scorer)
    pol = helpers.cuda_policy(c, objective, precision='bf16', scorer_config=cfg, sampling_propagation=sampling)
    pl = pol._ensure_planner()
    assert _choice(c, scorer_config=cfg)[0] == _lib.ROLLOUT_TC_WIDE_OBS
    pl_o = helpers.oracle_planner(c, objective, scorer_config=cfg, sampling_propagation=sampling)
    rng = np.random.default_rng(6)
    acts = rng.uniform(-1, 1, (c['N'], c['H'], c['A'])).astype(np.float32)
    eps = rng.standard_normal((c['H'], c['P'] * c['N'], c['O'])).astype(np.float32)
    B = c['P'] * c['N']
    ret = torch.full((B,), np.nan, dtype=torch.float32, device='cuda')
    mask = torch.full((B,), -1, dtype=torch.int64, device='cuda')
    csum = torch.full((B,), np.nan, dtype=torch.float32, device='cuda')
    d_state, d_acts, d_eps = dev(c['state'][None]), dev(acts[None]), dev(eps[None])
    _lib.check(lib.simba_rollout_score(pl, P(d_state), P(d_acts), P(d_eps), 0, 0, None, P(ret), P(mask),
                                       P(csum), None))
    torch.cuda.synchronize()
    traj, cum0, mask0, csum0 = _oracle_rows(c, pl_o, acts, eps, objective)
    got = ret.cpu().numpy()
    err = np.abs(got - cum0)
    agree = (mask.cpu().numpy().view(np.uint64) == mask0).mean()
    print("%s: max|dret| %.4g mean %.4g  mask agreement %.4f  cost rows %.3f  ret range [%.3f, %.3f]"
          % (name, err.max(), err.mean(), agree, (mask0 != 0).mean(), cum0.min(), cum0.max()))
    assert np.all(np.isfinite(got)) and np.all(np.isfinite(csum.cpu().numpy()))
    assert err.mean() < 1e-2
    assert agree > 1.0 - 0.002 * c['H']
    cand = np.abs(got.reshape(c['P'], c['N']).mean(0) - cum0.reshape(c['P'], c['N']).mean(0))
    assert cand.max() < 2e-2


# ---- 3: in-kernel noise vs the Philox counter contract -------------------------------------------------------
@pytest.mark.parametrize("obs", [92, 124])
def test_device_noise_follows_the_philox_contract(obs, monkeypatch):
    from simba_b200 import _lib
    c = _workload(obs, S=3)
    assert _choice(c) == (_lib.ROLLOUT_TC_WIDE_OBS, len(_tiles(c)))
    it = 3
    rng = np.random.default_rng(31)
    acts = rng.uniform(-1, 1, (c['S'], c['N'], c['H'], c['A'])).astype(np.float32)
    _set_switches(monkeypatch)
    dev_rows = _rollout(c, 'bf16', acts, None, SEED64, it)

    def compare(eps):
        ret, mask, csum = _rollout(c, 'bf16', acts, eps)
        return (np.abs(ret - dev_rows[0]).mean(), (mask == dev_rows[1]).mean(), (csum == dev_rows[2]).mean())

    good = compare(_contract_eps(c, SEED64, it))
    print("O=%d S=%d: contract mean|dret| %.3g, masks identical %.4f, cost sums identical %.4f" % (obs, c['S'], *good))
    assert np.all(np.isfinite(dev_rows[0]))
    assert good[0] <= NOISE_BOUNDS['mean_dret']
    assert good[1] >= NOISE_BOUNDS['mask_same'] and good[2] >= NOISE_BOUNDS['csum_same']
    for name, make in _controls(c, SEED64, it).items():
        bad = compare(make())
        print("  control %-22s mean|dret| %.3g  ratio %.3g" % (name, bad[0], bad[0] / max(good[0], 1e-12)))
        assert bad[0] >= 10 * good[0] and bad[0] > 0, name


# ---- 4: whole plans, bf16 against fp32 -------------------------------------------------------------------------
def test_plan_close_to_fp32_at_c1_dims():
    from simba_b200 import _lib, synthetic
    c = _workload(92, cfg='c1')
    cfg = SCORERS['goal4']
    assert _choice(c, scorer_config=cfg)[0] == _lib.ROLLOUT_TC_WIDE_OBS
    z, eps, zf = synthetic.make_draws(c['I'], 1, c['N'], c['H'], c['A'], c['P'], c['O'])
    res = {}
    for precision in ('fp32', 'bf16'):
        pol = helpers.cuda_policy(c, 'penalty', precision=precision, scorer_config=cfg)
        pol.set_external_draws(z, eps, zf)
        a, s = pol.do_generate_action(c['state'])
        res[precision] = (a, s, pol.buffer(_lib.BUF_MU).cpu().numpy(), pol.buffer(_lib.BUF_ELITE, torch.int32).cpu().numpy())
    a32, s32, mu32, el32 = res['fp32']
    a16, s16, mu16, el16 = res['bf16']
    overlap = len(set(el32) & set(el16)) / float(len(el32))
    print("O=92 bf16 vs fp32 plan: action %s vs %s, score %.4f vs %.4f, elite overlap %.2f, max|dmu| %.3g"
          % (a16, a32, s16, s32, overlap, np.abs(mu16 - mu32).max()))
    assert np.all(np.isfinite(a16)) and np.isfinite(s16)
    assert abs(s16 - s32) < 5e-2
    assert overlap >= 0.85                  # measured 0.93 on a B200 (148 SMs, 1000 W)


# ---- 5: bit-identical checks ------------------------------------------------------------------------------------
def _plan(c, monkeypatch, switches=(), draws=None, seed=None, **kw):
    from simba_b200 import _lib
    _set_switches(monkeypatch, *switches)
    pol = helpers.cuda_policy(c, 'penalty', precision='bf16', scorer_config=SCORERS['goal4'], **kw)
    if draws is not None:
        pol.set_external_draws(*draws)
    a, s = pol.do_generate_action(np.asarray(c['state'], np.float32).reshape(c['S'], c['O']), seed=seed)
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


def test_batched_plans_with_early_exit_equal_per_state_plans(monkeypatch):
    """Four O = 92 states whose tiles straddle states; a stddev threshold between the states' first-iteration
    stddev means stops some after one iteration and the rest later. Each state's plan equals a one-state plan
    on the same draws, bit for bit, and the diagnostic switches change nothing."""
    from simba_b200 import synthetic
    c = _workload(92, S=4, H=8, I=4, N=40)
    draws = synthetic.make_draws(c['I'], c['S'], c['N'], c['H'], c['A'], c['P'], c['O'], seed=5)
    first = _plan(dict(c, I=1), monkeypatch, draws=tuple(d[:1] if d.ndim == 5 else d for d in draws))
    means = first['sigma'].mean(1)
    thr = float(np.sort(means)[1:3].mean())
    base = _plan(c, monkeypatch, draws=draws, stddev_threshold=thr)
    print("sigma means after one iteration %s, threshold %.6f, iterations %s" % (means, thr, base['iters']))
    assert base['iters'].min() == 1 and base['iters'].max() > 1
    assert np.all(np.isfinite(base['score']))
    z, eps, zf = draws
    for s in range(c['S']):
        one = _plan(_one_state(c, s), monkeypatch, draws=(z[:, s:s + 1], eps[:, s:s + 1], zf[s:s + 1]),
                    stddev_threshold=thr)
        _assert_plans_equal(base, one, s)
    for sw in ('SIMBA_B200_NO_PDL', 'SIMBA_B200_NO_FUSE'):
        _assert_plans_equal(base, _plan(c, monkeypatch, (sw,), draws=draws, stddev_threshold=thr))


@pytest.mark.parametrize("obs", [92, 124])
def test_plans_without_pdl_or_fused_update_are_bit_identical(obs, monkeypatch):
    """Device Philox and the CUDA graph, three states."""
    c = _workload(obs, S=3)
    base = _plan(c, monkeypatch, seed=SEED64)
    for sw in ('SIMBA_B200_NO_PDL', 'SIMBA_B200_NO_FUSE'):
        _assert_plans_equal(base, _plan(c, monkeypatch, (sw,), seed=SEED64))
    assert not np.array_equal(base['action'], _plan(c, monkeypatch, seed=SEED64 + 1)['action'])


def test_recommitted_weights_reach_the_captured_planner():
    """New weights set on an already used planner (re-packed in place, graph re-captured) give the rows and
    the plan of a fresh planner built on them."""
    from simba_b200 import _lib, synthetic
    lib = _lib.load()
    c = _workload(92, U=200, L=3)
    cfg = SCORERS['goal4']
    pol = helpers.cuda_policy(c, 'penalty', precision='bf16', scorer_config=cfg)
    a1, _ = pol.do_generate_action(c['state'], seed=9)
    w2 = synthetic.make_weights(c['E'], c['L'], c['U'], c['O'], c['A'], seed=123)
    for e in range(c['E']):
        pol.model.model.ensemble[e].set_weights(w2[e])
    a2, s2 = pol.do_generate_action(c['state'], seed=9)
    fresh = helpers.cuda_policy(dict(c, weights=w2), 'penalty', precision='bf16', scorer_config=cfg)
    a3, s3 = fresh.do_generate_action(c['state'], seed=9)
    assert np.array_equal(a2, a3) and s2 == s3 and not np.array_equal(a1, a2)
    rng = np.random.default_rng(8)
    acts = dev(rng.uniform(-1, 1, (1, c['N'], c['H'], c['A'])).astype(np.float32))
    eps = dev(rng.standard_normal((1, c['H'], c['P'] * c['N'], c['O'])).astype(np.float32))
    rows = []
    for p in (pol, fresh):
        B = c['P'] * c['N']
        out = [torch.empty(B, dtype=torch.float32, device='cuda'), torch.empty(B, dtype=torch.int64, device='cuda'),
               torch.empty(B, dtype=torch.float32, device='cuda')]
        _lib.check(lib.simba_rollout_score(p._ensure_planner(), P(dev(c['state'][None])), P(acts), P(eps), 0, 0,
                                           None, *[P(x) for x in out], None))
        torch.cuda.synchronize()
        rows.append([x.cpu().numpy() for x in out])
    for x, y in zip(*rows):
        assert np.array_equal(x, y)


SHARDED = r'''
import os, sys
sys.path[:0] = [sys.argv[1], os.path.join(sys.argv[1], 'ethz-safe-learning_b200')]
import numpy as np, torch, torch.distributed as dist
from simba_b200 import _lib, distributed as sd, synthetic
from tests.test_gpu_tc_obs_wide import GOAL4, SCORERS
rank, world = int(os.environ['RANK']), int(os.environ['WORLD_SIZE'])
torch.cuda.set_device(int(os.environ['LOCAL_RANK']))
dist.init_process_group('nccl', device_id=torch.device('cuda', int(os.environ['LOCAL_RANK'])))
c = synthetic.make_workload('c1', sensors=GOAL4, N=160, K=16)
single = synthetic.build_policy(c, 'penalty', precision='bf16', scorer_config=SCORERS['goal4'])
a1, s1 = single.do_generate_action(c['state'], seed=77)
el1 = single.buffer(_lib.BUF_ELITE, torch.int32).cpu().numpy()
shard = synthetic.build_policy(c, 'penalty', precision='bf16', scorer_config=SCORERS['goal4'], rank=rank,
                               world_size=world)
sd.init_population_sharding(shard)
a2, s2 = shard.do_generate_action(c['state'], seed=77)
el2 = shard.buffer(_lib.BUF_ELITE, torch.int32).cpu().numpy()
t = torch.tensor([1.0 if (np.array_equal(a1, a2) and s1 == s2 and np.array_equal(el1, el2)) else 0.0], device='cuda')
dist.all_reduce(t, op=dist.ReduceOp.MIN)
if rank == 0:
    print("O=92 sharded plan equals the single-GPU plan on every rank: %s" % bool(t.item() > 0))
dist.destroy_process_group()
'''


def test_population_sharded_plan_equals_single_gpu_plan(tmp_path):
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs (have %d)" % n)
    script = tmp_path / 'sharded_obs_wide.py'
    script.write_text(SHARDED)
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2',
           '--master-addr', '127.0.0.1', '--master-port', '29633', str(script), ROOT]
    out = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
    sys.stdout.write(out.stdout[-3000:])
    assert out.returncode == 0, out.stderr[-3000:]
    assert "equals the single-GPU plan on every rank: True" in out.stdout
