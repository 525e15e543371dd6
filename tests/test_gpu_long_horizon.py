"""Planning horizons beyond 64 steps. A row's cost history (bit t = cost(s_t) * (1 - done_t)) is W = ceil(H / 64)
64-bit words stored as planes [W, S, P, N_local]: plane w holds steps [64 w, 64 w + 64), plane 0 is the whole
history for H <= 64. Workloads use var-head bias -5 (sigma ~ 0.08 per step), as the parity tests of the unfold
kernels do, and observe the goal distance (a 39-dim layout: goal_dist at index 3, hazards and vases lidars) rather than
the goal lidar: on PointGoal1's layout every row of these synthetic models reaches the goal within 64 steps, after
which its cost bits are masked, so no plane beyond the first would carry a bit.

  1  fp32 rows against the oracle on external draws, H in {65, 100, 128, 200}, every objective: each mask word
     equal on rows whose hard decisions are not within 1e-4 of a threshold up to that word's last step, returns
     within the 1e-4 contract, cost sums exact; score_reduce and compute_objective on the planes
  2  fp32 whole plans against the oracle at H = 100: elite sets exact, mu / sigma within 1e-4
  3  every bf16 form at H > 64 against the fp32 kernel (tolerances below, measured on a B200), and the diagnostic
     switches NO_PAIR / NO_TAIL_SPLIT bit-identical
  4  fused vs separate update bit-identical (SIMBA_B200_NO_FUSE), batched plans with early exit equal per-state plans
  5  two GPUs: the population-sharded plan at H = 100 equals the one-GPU plan bit for bit
  6  boundaries: H = 64 keeps one plane and its launch count, H = 65 and H * A = 1024 are accepted, 1025 is not
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import simba_oracle as so
from tests import helpers

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SWITCHES = ('SIMBA_B200_NO_PAIR', 'SIMBA_B200_NO_FUSE', 'SIMBA_B200_NO_PDL', 'SIMBA_B200_NO_TAIL_SPLIT')


def _lib():
    from simba_b200 import _lib as L
    return L


def _dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _P(t):
    return C.c_void_p(0 if t is None else t.data_ptr())


def _planes(H):
    return (H + 63) // 64


def _set_switches(monkeypatch, *on):
    for name in SWITCHES:
        if name in on:
            monkeypatch.setenv(name, '1')
        else:
            monkeypatch.delenv(name, raising=False)


GD_SENSORS = dict(accelerometer=3, goal_dist=1, hazards_lidar=16, vases_lidar=16, velocimeter=3)
GD_SCORER = dict(observe_goal_lidar=False, observe_goal_dist=True, constrain_vases=True)
# the same at PointGoal1's width (60 dims: goal_dist at index 24). The CTA-pair forms run on this one: on the 39-dim
# layout the pair kernel's rows differ from one CTA's at every horizon, H <= 64 included (DESIGN.md section 7)
GD60_SENSORS = dict(accelerometer=3, aux=21, goal_dist=1, hazards_lidar=16, vases_lidar=16, velocimeter=3)


def _workload(cfg='tiny', sensors=GD_SENSORS, **over):
    return helpers.workload(cfg, sensors=sensors, var_bias=-5.0, **over)


def _oracle_rows(c, pl_o, acts, eps, objective):
    """Per-row (trajectories, return, cost-mask planes [W, P*N], cost sum) of the oracle's trajectories."""
    P_, N, H = c['P'], c['N'], c['H']
    acts_b = np.tile(acts, (P_, 1, 1))
    s0 = np.broadcast_to(c['state'], (P_ * N, c['O']))
    traj = pl_o.model.unfold_sequences(s0, acts_b, eps, pl_o.member_of_row())
    B = P_ * N
    cum = np.zeros(B, np.float32); done = np.zeros(B, bool); csum = np.zeros(B, np.float32)
    planes = np.zeros((_planes(H), B), np.uint64)
    done_first = objective in ('penalty', 'feasible_first')
    for t in range(H):
        r, d = pl_o.reward(traj[:, t], None, traj[:, t + 1])
        cost = pl_o.cost(traj[:, t], None, traj[:, t + 1])
        if done_first:
            done = done | d
        bit = ((cost > 0) & ~done).astype(np.uint64) << np.uint64(t % 64)
        cum = cum + r * (1 - done.astype(np.float32))
        planes[t // 64] |= bit
        if not done_first:
            done = done | d
        csum = csum + cost
    return traj, cum, planes, csum


def _first_fragile(c, traj, scorer_config=GD_SCORER):
    """Per row, the first state index whose goal or constraint decision is within 1e-4 of its threshold in the
    oracle (H + 1 when none is): from there on the row's bits may legitimately differ."""
    sc = so.Scorer(scorer_config, c['table'])
    first = np.full(traj.shape[0], c['H'] + 1)
    for t in range(c['H'] + 1, 0, -1):
        x = traj[:, t - 1]
        frag = np.abs(sc.goal_distance_metric(x) - np.float32(sc.c['goal_size'] * 0.8)) < 1e-4
        for name in ('vases', 'hazards', 'pillars', 'gremlins'):
            if sc.c['constrain_' + name]:
                d = sc.closest_distance(x[:, c['table'][name + '_lidar']])
                frag |= np.abs(d - np.float32(sc.c[name + '_size'])) < 1e-4
        first[frag] = t - 1
    return first


def _rollout(c, precision, objective, acts, eps, scorer_config=GD_SCORER, seed=0):
    """One simba_rollout_score call on a fresh planner: acts [S, N, H, A], eps [S, H, P*N, O] or None (device Philox
    with this seed) -> (return [S, P*N], mask planes [W, S, P*N] uint64, cost sum [S, P*N], policy, rollout kernel)."""
    L = _lib()
    lib = L.load()
    pol = helpers.cuda_policy(c, objective, precision=precision, scorer_config=scorer_config)
    pl = pol._ensure_planner()
    S, B, W = c['S'], c['P'] * c['N'], _planes(c['H'])
    ret = torch.full((S * B,), np.nan, dtype=torch.float32, device='cuda')
    mask = torch.full((W * S * B,), -1, dtype=torch.int64, device='cuda')
    csum = torch.full((S * B,), np.nan, dtype=torch.float32, device='cuda')
    d_state = _dev(np.asarray(c['state'], np.float32).reshape(S, c['O']))
    d_acts = _dev(acts)
    d_eps = _dev(eps) if eps is not None else None
    L.check(lib.simba_rollout_score(pl, _P(d_state), _P(d_acts), _P(d_eps), seed, 0, None, _P(ret), _P(mask),
                                    _P(csum), None))
    torch.cuda.synchronize()
    kernel, items = C.c_int32(-1), C.c_int32(-1)
    L.check(lib.simba_planner_rollout_kernel(pl, C.byref(kernel), C.byref(items)))
    return (ret.cpu().numpy().reshape(S, B), mask.cpu().numpy().view(np.uint64).reshape(W, S, B),
            csum.cpu().numpy().reshape(S, B), pol, kernel.value)


def _max_counts(planes, P_, N, H):
    """max_t of the per-step particle counts of the set bits, per candidate: planes [W, P*N]."""
    bits = np.zeros((P_ * N, H), np.int64)
    for t in range(H):
        bits[:, t] = (planes[t // 64] >> np.uint64(t % 64)) & np.uint64(1)
    return bits.reshape(P_, N, H).sum(0).max(-1).astype(np.float32)


# ---- 1: fp32 rows against the oracle ----------------------------------------------------------------------------
@pytest.mark.parametrize("objective", ['reward', 'penalty', 'least_cost', 'feasible_first'])
@pytest.mark.parametrize("H", [65, 100, 128, 200])
def test_fp32_rows_match_oracle_in_planes(H, objective):
    L = _lib()
    lib = L.load()
    c = _workload(H=H)
    P_, N, B, W = c['P'], c['N'], c['P'] * c['N'], _planes(H)
    rng = np.random.default_rng(60 + H)
    acts = rng.uniform(-1, 1, (c['N'], H, c['A'])).astype(np.float32)
    eps = rng.standard_normal((H, B, c['O'])).astype(np.float32)
    ret, planes, csum, pol, _ = _rollout(c, 'fp32', objective, acts[None], eps[None])
    ret, planes, csum = ret[0], planes[:, 0], csum[0]
    pl_o = helpers.oracle_planner(c, objective, scorer_config=GD_SCORER)
    traj, cum0, planes0, csum0 = _oracle_rows(c, pl_o, acts, eps, objective)
    first = _first_fragile(c, traj)
    ok = first > H
    print("H=%d %s: fragile rows %.3f, max|dret| %.3g on the others, rows with cost bits per plane %s"
          % (H, objective, 1 - ok.mean(), np.abs(ret - cum0)[ok].max(), (planes0 != 0).mean(1)))
    assert ok.mean() > 0.9
    for w in range(W):
        okw = first > min(64 * w + 64, H)          # the states this word's steps read are all clear of a threshold
        assert np.array_equal(planes[w][okw], planes0[w][okw]), w
    assert (planes0[W - 1] != 0).any() and len(np.unique(planes0[W - 1])) > 1      # bits beyond step 64
    assert np.allclose(ret[ok], cum0[ok], rtol=1e-4, atol=2e-5)
    assert np.array_equal(csum[ok], csum0[ok])
    # the reduction runs over every plane: cost = max_t count_t (penalty, feasible_first), mean cost sum
    # (least_cost), 0 (reward); return = mean over particles in particle order
    pairs = torch.zeros((N, 2), dtype=torch.float32, device='cuda')
    d_ret, d_mask, d_csum = _dev(ret), _dev(planes.view(np.int64)), _dev(csum)
    L.check(lib.simba_score_reduce(pol._ensure_planner(), _P(d_ret), _P(d_mask), _P(d_csum), None, _P(pairs), None))
    pairs = pairs.cpu().numpy()
    mean_ret = np.zeros(N, np.float32)
    mean_csum = np.zeros(N, np.float32)
    for p in range(P_):
        mean_ret += ret[p * N:(p + 1) * N]
        mean_csum += csum[p * N:(p + 1) * N]
    assert np.array_equal(pairs[:, 0], mean_ret / np.float32(P_))
    want = {'reward': np.zeros(N, np.float32), 'least_cost': mean_csum / np.float32(P_)}.get(
        objective, _max_counts(planes, P_, N, H))
    assert np.array_equal(pairs[:, 1], want)
    # compute_objective on materialised [P*N, H+1, O] trajectories: the oracle's (return, cost) pairs
    scores = torch.zeros(N, dtype=torch.float32, device='cuda')
    tp = torch.zeros((N, 2), dtype=torch.float32, device='cuda')
    d_traj = _dev(traj.astype(np.float32))
    L.check(lib.simba_score_trajectories(pol._ensure_planner(), _P(d_traj), _P(scores), _P(tp), None))
    _, ret_o, cost_o = pl_o.compute_scores(traj.astype(np.float32), np.tile(acts, (P_, 1, 1)))
    tp = tp.cpu().numpy()
    assert np.allclose(tp[:, 0], ret_o, rtol=1e-6, atol=1e-6) and np.array_equal(tp[:, 1], cost_o.astype(np.float32))
    assert pol.compute_objective(traj.astype(np.float32)).shape == (N,)


# ---- 2: fp32 whole plans against the oracle --------------------------------------------------------------------
@pytest.mark.parametrize("objective", ['penalty', 'feasible_first'])
def test_fp32_plan_matches_oracle_at_h100(objective):
    from simba_b200 import synthetic
    L = _lib()
    c = _workload(H=100)
    z, eps, zf = synthetic.make_draws(c['I'], 1, c['N'], c['H'], c['A'], c['P'], c['O'])
    pol = helpers.cuda_policy(c, objective, precision='fp32', scorer_config=GD_SCORER)
    pol.set_external_draws(z, eps, zf)
    action, score = pol.do_generate_action(c['state'])
    tr = so.Trace()
    a0, s0, n0 = helpers.oracle_planner(c, objective, scorer_config=GD_SCORER).do_generate_action(c['state'], z[:, 0], eps[:, 0], zf[0], tr)
    assert np.array_equal(pol.buffer(L.BUF_ELITE, torch.int32).cpu().numpy(), tr[-1]['elite'])
    mu = pol.buffer(L.BUF_MU).cpu().numpy().reshape(c['H'], c['A'])
    sg = pol.buffer(L.BUF_SIGMA).cpu().numpy().reshape(c['H'], c['A'])
    assert np.allclose(mu, tr[-1]['mu'], rtol=1e-4, atol=1e-6) and np.allclose(sg, tr[-1]['sigma'], rtol=1e-4, atol=1e-6)
    assert np.allclose(action, a0, rtol=1e-4, atol=1e-6) and np.isclose(score, s0, rtol=1e-4, atol=1e-5)
    assert max(t['cost'].max() for t in tr) > 0                 # the counts are exercised


# ---- 3: every bf16 form at H > 64 against the fp32 kernel --------------------------------------------------------
# Tolerances of the bf16 rows against the fp32 kernel's on the same external draws, per form and horizon: mean
# |d return| <= ret, at least `agree` of the rows have every mask word equal, and at least `late` of the fp32 rows
# carry cost bits beyond step 64 (so that the later planes are compared on real bits). Measured on a B200 (1000 W
# power limit), in brackets: the rows drift apart with the horizon (bf16 weights, activations and draws at every step
# of trajectories that keep hitting hazards). The 1 - 0.002 H rule of the H <= 64 tests says nothing at H = 256.
FORMS = {  # name: (workload, overrides, switches, kernel constant name, sensors, scorer config, ret, agree, late)
    'one-cta': ('tiny', dict(H=100), ('SIMBA_B200_NO_PAIR',), 'ROLLOUT_TC_ONE_CTA', None, None,
                4e-3, 0.985, 0.8),                                              # [2.2e-3, 0.995, 0.875]
    'pair': ('tiny', dict(H=128), (), 'ROLLOUT_TC_PAIR', 'gd60', None,
             8e-3, 0.98, 0.4),                                                  # [4.8e-3, 0.990, 0.443]
    'pair-h256': ('tiny', dict(H=256), (), 'ROLLOUT_TC_PAIR', 'gd60', None,
                  2.5e-2, 0.88, 0.4),                                           # [1.7e-2, 0.896, 0.427]
    'two-tile': ('c1', dict(H=100, S=16), (), 'ROLLOUT_TC_TWO_TILE', None, None,   # Philox draws (eps: 1 GB)
                 3e-3, 0.98, 0.25),                                             # [1.6e-3, 0.989, 0.279]
    'wide64': ('c5', dict(H=100), (), 'ROLLOUT_TC_WIDE', None, None,
               4e-3, 0.975, 0.55),                                              # [2.2e-3, 0.984, 0.631]
    'wide128': ('tiny', dict(H=100), (), 'ROLLOUT_TC_WIDE_OBS', 'goal_dist', 'goal_dist',   # obs 100, goal_dist at 67
                1e-3, 0.995, 0.12),                                             # [5.6e-4, 1.000, 0.130]
}


def _form_workload(name):
    cfg, over, switches, kernel, sensors, scorer = FORMS[name][:6]
    if sensors == 'gd60':
        return _workload(cfg, sensors=GD60_SENSORS, **over), switches, kernel, GD_SCORER
    if sensors is not None:
        from tests.test_gpu_tc_obs_wide import SCORERS, SENSORS
        return _workload(cfg, sensors=SENSORS[sensors], **over), switches, kernel, SCORERS[scorer]
    return _workload(cfg, **over), switches, kernel, GD_SCORER


@pytest.mark.parametrize("name", list(FORMS))
def test_bf16_forms_hold_against_fp32_beyond_64_steps(name, monkeypatch):
    L = _lib()
    c, switches, kernel, scorer = _form_workload(name)
    H, S, B = c['H'], c['S'], c['P'] * c['N']
    rng = np.random.default_rng(7)
    acts = rng.uniform(-1, 1, (S, c['N'], H, c['A'])).astype(np.float32)
    eps = rng.standard_normal((S, H, B, c['O'])).astype(np.float32) if name != 'two-tile' else None
    W = _planes(H)

    def rows(precision):
        r, m, cs, _, k = _rollout(c, precision, 'penalty', acts, eps, scorer, seed=21)
        return r.reshape(-1), m.reshape(W, -1), cs.reshape(-1), k
    _set_switches(monkeypatch, *switches)
    r16, m16, c16, k16 = rows('bf16')
    assert k16 == getattr(L, kernel), (k16, kernel)
    _set_switches(monkeypatch)
    r32, m32, c32, k32 = rows('fp32')
    assert k32 == L.ROLLOUT_FP32
    dret = np.abs(r16 - r32).mean()
    agree = (m16 == m32).all(0).mean()
    late = (m32[1:] != 0).any(0).mean()                       # rows with cost bits beyond step 64
    print("%s H=%d: mean|dret| %.4g max %.4g, rows with every mask word equal %.4f, per plane %s, rows with bits "
          "beyond step 64 %.3f" % (name, H, dret, np.abs(r16 - r32).max(), agree, (m16 == m32).mean(1), late))
    assert np.all(np.isfinite(r16)) and np.all(np.isfinite(c16))
    ret_tol, agree_min, late_min = FORMS[name][6:]
    assert late >= late_min                                   # the later planes are compared on real bits
    assert dret <= ret_tol
    assert agree >= agree_min
    # the diagnostic switches: the pair kernel equals one CTA, the two-tile kernel is unchanged without its tail split
    other = {'pair': ('SIMBA_B200_NO_PAIR',), 'pair-h256': ('SIMBA_B200_NO_PAIR',),
             'two-tile': ('SIMBA_B200_NO_TAIL_SPLIT',)}.get(name)
    if other is not None:
        _set_switches(monkeypatch, *other)
        r2, m2, c2, k2 = rows('bf16')
        _set_switches(monkeypatch)
        if name != 'two-tile':
            assert k2 == L.ROLLOUT_TC_ONE_CTA
        assert np.array_equal(r2, r16) and np.array_equal(m2, m16) and np.array_equal(c2, c16)


# ---- 4: fused vs separate update, batched vs per-state plans ----------------------------------------------------
def _plan(c, monkeypatch, switches=(), draws=None, seed=None, precision='bf16', **kw):
    L = _lib()
    _set_switches(monkeypatch, *switches)
    pol = helpers.cuda_policy(c, 'penalty', precision=precision, scorer_config=GD_SCORER, **kw)
    if draws is not None:
        pol.set_external_draws(*draws)
    states = np.asarray(c['state'], np.float32).reshape(c['S'], c['O'])
    a, s = pol.do_generate_action(states, seed=seed)
    S = c['S']
    out = dict(action=np.asarray(a).reshape(S, -1), score=np.asarray(s).reshape(S),
               iters=np.asarray(pol.iterations_run).reshape(S).copy(),
               mu=pol.buffer(L.BUF_MU).cpu().numpy().reshape(S, -1),
               sigma=pol.buffer(L.BUF_SIGMA).cpu().numpy().reshape(S, -1),
               elite=pol.buffer(L.BUF_ELITE, torch.int32).cpu().numpy().reshape(S, -1))
    launches = pol.launches_per_plan
    _set_switches(monkeypatch)
    return out, launches


def _assert_plans_equal(a, b, s=None):
    for k in a:
        x = a[k] if s is None else a[k][s:s + 1]
        assert np.array_equal(x, b[k]), (k, s)


@pytest.mark.parametrize("case", ['staged', 'unstaged', 'c1-fp32'])
def test_fused_update_equals_separate_kernels_at_h100(case, monkeypatch):
    """The fused update stages the W mask planes in shared memory and counts steps plane by plane where the
    staging fits (a small population), and reads them from global memory otherwise (C1 dims): both are bit-identical
    to the separate reduce / select / refit kernels."""
    from simba_b200 import synthetic
    over = dict(staged=dict(N=32, K=6, P=8), unstaged=dict(), **{'c1-fp32': dict()})[case]
    c = _workload('tiny' if case == 'staged' else 'c1', H=100, **over)
    precision = 'fp32' if case == 'c1-fp32' else 'bf16'
    draws = synthetic.make_draws(c['I'], 1, c['N'], c['H'], c['A'], c['P'], c['O'], seed=11)
    fused, n_fused = _plan(c, monkeypatch, draws=draws, precision=precision)
    separate, n_sep = _plan(c, monkeypatch, ('SIMBA_B200_NO_FUSE',), draws=draws, precision=precision)
    print("%s: launches fused %d, separate %d, score %s" % (case, n_fused, n_sep, fused['score']))
    assert n_fused == 1 + 2 * c['I'] and n_sep == 5 * c['I'] + 3
    _assert_plans_equal(fused, separate)
    # production mode (device Philox)
    _assert_plans_equal(_plan(c, monkeypatch, seed=5, precision=precision)[0],
                        _plan(c, monkeypatch, ('SIMBA_B200_NO_FUSE',), seed=5, precision=precision)[0])


def test_batched_plans_with_early_exit_equal_per_state_plans_at_h100(monkeypatch):
    """Four states, a stddev threshold between their first-iteration stddev means: two stop after one iteration,
    two run on. Every state's plan equals a one-state plan on the same draws, fused and separate alike."""
    from simba_b200 import synthetic
    S = 4
    c = _workload('tiny', H=100, S=S, I=4)
    z, eps, zf = synthetic.make_draws(c['I'], S, c['N'], c['H'], c['A'], c['P'], c['O'], seed=5)
    states = np.asarray(c['state'], np.float32).reshape(S, -1)

    def one(s, **kw):
        return dict(c, S=1, state=states[s], **kw)
    first = sorted(_plan(one(s, I=1), monkeypatch, draws=(z[:1, s:s + 1], eps[:1, s:s + 1], zf[s:s + 1]))[0]
                   ['sigma'].mean() for s in range(S))
    thr = float((first[1] + first[2]) / 2)
    base, _ = _plan(c, monkeypatch, draws=(z, eps, zf), stddev_threshold=thr)
    print("first-iteration stddev means %s, threshold %.5f, iterations %s" % (first, thr, base['iters']))
    assert base['iters'].min() == 1 and base['iters'].max() > 1
    for s in range(S):
        got, _ = _plan(one(s), monkeypatch, draws=(z[:, s:s + 1], eps[:, s:s + 1], zf[s:s + 1]), stddev_threshold=thr)
        _assert_plans_equal(base, got, s)
    _assert_plans_equal(base, _plan(c, monkeypatch, ('SIMBA_B200_NO_FUSE',), draws=(z, eps, zf),
                                    stddev_threshold=thr)[0])


# ---- 5: two GPUs -----------------------------------------------------------------------------------------------
def test_population_sharded_plan_equals_single_gpu_plan_at_h100():
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs (have %d)" % n)
    code = r'''
import os, sys
sys.path[:0] = [%r, os.path.join(%r, 'ethz-safe-learning_b200')]
import numpy as np, torch, torch.distributed as dist
from simba_b200 import _lib, distributed as sd, synthetic
rank, world = int(os.environ['RANK']), int(os.environ['WORLD_SIZE'])
torch.cuda.set_device(int(os.environ['LOCAL_RANK']))
dist.init_process_group('nccl', device_id=torch.device('cuda', int(os.environ['LOCAL_RANK'])))
ok = True
for precision in ('fp32', 'bf16'):
    c = synthetic.make_workload('c1', N=160, K=16, H=100, var_bias=-5.0, sensors=%r)
    single = synthetic.build_policy(c, 'penalty', precision=precision, scorer_config=%r)
    a1, s1 = single.do_generate_action(c['state'], seed=77)
    mu1 = single.buffer(_lib.BUF_MU).cpu().numpy(); el1 = single.buffer(_lib.BUF_ELITE, torch.int32).cpu().numpy()
    shard = synthetic.build_policy(c, 'penalty', precision=precision, rank=rank, world_size=world,
                                   scorer_config=%r)
    sd.init_population_sharding(shard)
    a2, s2 = shard.do_generate_action(c['state'], seed=77)
    mu2 = shard.buffer(_lib.BUF_MU).cpu().numpy(); el2 = shard.buffer(_lib.BUF_ELITE, torch.int32).cpu().numpy()
    same = np.array_equal(a1, a2) and s1 == s2 and np.array_equal(mu1, mu2) and np.array_equal(el1, el2)
    t = torch.tensor([1.0 if same else 0.0], device='cuda')
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("[%%s] H=100 sharded == single-GPU plan on every rank: %%s" %% (precision, bool(t.item() > 0)))
    ok = ok and bool(t.item() > 0)
dist.destroy_process_group()
sys.exit(0 if ok else 1)
''' % (ROOT, ROOT, GD60_SENSORS, GD_SCORER, GD_SCORER)
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        script = os.path.join(d, 'sharded_h100.py')
        with open(script, 'w') as f:
            f.write(code)
        cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2',
               '--master-addr', '127.0.0.1', '--master-port', '29641', script]
        out = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
    sys.stdout.write(out.stdout[-3000:])
    assert out.returncode == 0, out.stderr[-3000:]
    assert out.stdout.count("sharded == single-GPU plan on every rank: True") == 2


# ---- 6: boundaries ---------------------------------------------------------------------------------------------
def test_horizon_boundaries():
    from simba_b200 import SimbaError
    L = _lib()
    sizes = {}
    for H in (64, 65, 512):                         # 512 * A = 1024 (A = 2): the largest plan accepted
        c = _workload(H=H)
        pol = helpers.cuda_policy(c, 'penalty', precision='bf16', scorer_config=GD_SCORER)
        p, n = C.c_void_p(), C.c_uint64()
        L.check(L.load().simba_planner_buffer(pol._ensure_planner(), L.BUF_ROW_COSTMASK, C.byref(p), C.byref(n)))
        sizes[H] = n.value
        a, s = pol.do_generate_action(c['state'], seed=3)
        assert np.all(np.isfinite(a)) and np.isfinite(s)
        assert pol.launches_per_plan == 1 + 2 * c['I']           # the fused update
    plane = 8 * c['P'] * c['N']                     # bytes of one plane: one state, one rank
    assert sizes == {64: plane, 65: 2 * plane, 512: 8 * plane}
    assert L.SIMBA_MAX_HORIZON == 1024
    c = _workload(H=1024, A=1)                      # 1024 * 1
    pol = helpers.cuda_policy(c, 'penalty', precision='fp32', scorer_config=GD_SCORER)
    a, s = pol.do_generate_action(c['state'], seed=3)
    assert np.all(np.isfinite(a)) and np.isfinite(s)
    for over in (dict(H=1025, A=1), dict(H=205, A=5), dict(H=513, A=2)):       # H * A = 1025, 1025, 1026
        c = _workload(**over)
        with pytest.raises(SimbaError) as e:
            helpers.cuda_policy(c, 'penalty', precision='fp32', scorer_config=GD_SCORER)._ensure_planner()
        assert e.value.code == -1, over


def test_h64_plans_keep_one_plane_and_the_c1_launch_count():
    """H <= 64 keeps its layout and kernels: C1 at H = 64 runs the same number of launches as at H = 15, and a plan at
    C1 dims up to H = 256 keeps the fused update."""
    for H, n in ((15, 11), (64, 11), (65, 11), (256, 11)):
        c = _workload('c1', H=H)
        pol = helpers.cuda_policy(c, 'penalty', precision='bf16', scorer_config=GD_SCORER)
        assert pol.launches_per_plan == n, (H, pol.launches_per_plan)


def test_python_policies_plan_beyond_64_steps():
    """CemMpc, SafeCemMpc and RandomShootingMpc take horizon > 64 as they are: finite, reproducible plans."""
    from simba_b200.policies import RandomShootingMpc
    c = _workload(H=130)
    for objective in ('reward', 'penalty'):
        pol = helpers.cuda_policy(c, objective, precision='bf16', scorer_config=GD_SCORER)
        a1, s1 = pol.do_generate_action(c['state'], seed=9)
        a2, s2 = pol.do_generate_action(c['state'], seed=9)
        assert np.all(np.isfinite(a1)) and np.array_equal(a1, a2) and s1 == s2
    base = helpers.cuda_policy(c, 'reward', precision='fp32', scorer_config=GD_SCORER)
    rs = RandomShootingMpc(base.model, base.environment, c['H'], None, c['N'], c['P'], precision='fp32', seed=1)
    a, s = rs.do_generate_action(c['state'])
    assert a.shape == (c['A'],) and np.all(np.isfinite(a)) and np.isfinite(s)
